#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json): Mrays/s (primary + secondary).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config C1|C2|C3|C5] [--no-extras] [--dump-outputs DIR]

Default workload = BASELINE config C2: procedural ~1M-triangle displaced mesh in an emitter-lit room, 1920x1080, 1 spp per pass,
depth 8 (bounces = 6), GGX + diffuse.  A step = one progressive pass over the whole frame.  N>1 (torchrun, one rank per GPU): the scene
and its BVH are replicated, rank r renders sample s = step*N + r of every pixel (weak scaling: one full-frame pass per GPU per step), and
the accumulation buffers are combined by one NCCL reduce per pass — behind the C ABI (rtx_comm_init / rtx_reduce_accum), on a side
stream, overlapped with the next pass (SURVEY.md §8e).

One JSON line on rank 0:
  value        rays/s with everything resident in HBM (CUDA events on the engine's stream, max over ranks)
  e2e          the same metric through the C ABI with HOST buffers (instance + camera upload, render, RGBA8 read-back per step)
  roofline     achieved algorithmic GB/s of the closest-hit traversal kernel against the measured HBM peak
  cpu_baseline the CPU oracle (oracle/: a port of the reference's shaders, pinned to their text by tests/test_ref_pins.py), one thread,
               on a bounded pixel subsample of the same workload
  parity       the GPU accumulation of one sample bit-compared with the oracle image of that cpu_baseline sample, plus hit ids
  configs      (N=1, default config) compact runs of the other BASELINE configs C1, C3, C5 with their own roofline + parity
  c4_strong    BASELINE config C4 (4K progressive render split by samples over the N GPUs, one reduce per pass): strong scaling
`--dump-outputs DIR` writes, after the timed steps, what the timed path computed in its last step, at most 64 MB in all: for a render
config accum.npy (gPermanentData, H x W x 4 float32; above 2^21 pixels, as C3's 3840x2160, a fixed, seeded sample of pixels, n x 4,
with their row-major indices in accum_rows.npy) and counters.npy (closest rays, shadow rays, paths of the timed steps); for C5 the hit
records (t, u, v, prim, inst as float64) of a fixed, seeded sample of each batch, with the sampled rows.  The inputs are seeded: two
builds run with the same arguments can be compared array by array.  Except C5's incoherent batch: its rays start at the coherent
batch's hit points and only rays that hit are kept, so a build whose coherent t differs in any bit traces other incoherent rays, and
its sampled rows are drawn from a batch of another size; compare hits_incoherent row by row only where hits_coherent agree exactly.
`--impl reference` times the CPU port on all host threads (the reference itself is a Windows/DX12 application and cannot run); it loads
no engine library and prints the same `config`.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mrays/s (primary+secondary)"
UNIT = "Mrays/s"
FLAG_JITTER, FLAG_LAMBERT_ONLY = 1, 2


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="C2", choices=["C1", "C2", "C3", "C5"])
    ap.add_argument("--width", type=int, default=0, help="override the config's width")
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--side", type=int, default=296, help="C2 cube-sphere side: 12*side^2 triangles (296 -> 1,051,392)")
    ap.add_argument("--tris", type=int, default=1_000_000, help="C5 scene size")
    ap.add_argument("--bounces", type=int, default=-1, help="override the config's path length")
    ap.add_argument("--cpu-step", type=int, default=0, help="pixel subsampling of the CPU legs (every n-th pixel in x and y); 0 = per config")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the compact runs of the other BASELINE configs and C4")
    ap.add_argument("--c4-spp", type=int, default=16, help="samples per pixel of one C4 step (split over the ranks)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the timed path computed in its last step as DIR/<name>.npy (rank 0)")
    return ap.parse_args()


DUMP_MAX_BYTES = 64 * 10 ** 6      # everything --dump-outputs writes in one run
DUMP_SAMPLE_PIXELS = 1 << 21       # accumulation pixels kept when the whole buffer would not fit (32 MB float32 + 16 MB indices)
DUMP_SAMPLE_RAYS = 1 << 19         # hit records kept per C5 batch (2 x (20 MB float64 + 4 MB indices))
_dumped_bytes = 0


def dump_outputs(d, arrays):
    """Writes {name: array} as d/<name>.npy in float32 or float64, so that two builds can be compared output by output."""
    global _dumped_bytes
    arrays = {name: np.asarray(a) for name, a in arrays.items()}
    arrays = {name: a if a.dtype in (np.float32, np.float64) else a.astype(np.float64) for name, a in arrays.items()}
    _dumped_bytes += sum(a.nbytes for a in arrays.values())
    if _dumped_bytes > DUMP_MAX_BYTES:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes, more than %d" % (_dumped_bytes, DUMP_MAX_BYTES))
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a)


def seeded_rows(n, k):
    """A fixed sample of k of n row indices (all of them when k >= n), in ascending order."""
    return np.arange(n) if k >= n else np.sort(np.random.RandomState(0).choice(n, k, replace=False))


def hit_records(h):
    """rtx_trace_device's 5-word hit records (t, u, v as float32; prim, inst as uint32) as float64 columns."""
    h = np.ascontiguousarray(h, dtype=np.float32)
    return np.concatenate([h[:, :3].astype(np.float64), h[:, 3:].view(np.uint32).astype(np.float64)], axis=1)


# ------------------------------------------------------------------------------------------------ workloads (BASELINE.json configs)
def config_of(name, args):
    if name == "C1":
        c = dict(kind="render", W=256, H=256, bounces=2, flags=FLAG_JITTER | FLAG_LAMBERT_ONLY, spp=16, cpu_step=1,
                 scene=lambda r: r.scenes.cornell(), label="C1 %s 256x256 16 spp/pass depth 4 (bounces=2) Lambert only, jitter")
    elif name == "C2":
        c = dict(kind="render", W=1920, H=1080, bounces=6, flags=0, spp=1, cpu_step=2,
                 scene=lambda r: r.scenes.mesh_room(n=args.side, seed=1), label="C2 %s %dx%d 1spp/pass depth %d (bounces=%d) GGX+diffuse")
    elif name == "C3":
        c = dict(kind="render", W=3840, H=2160, bounces=3, flags=0, spp=1, cpu_step=8,
                 scene=lambda r: r.scenes.instanced_blobs(), label="C3 %s %dx%d 1spp/pass depth %d (bounces=%d) 1000 instances, emissive instances with NEE")
    else:
        c = dict(kind="trace", W=4096, H=4096, bounces=0, flags=0, spp=1, cpu_step=16,
                 scene=lambda r: r.scenes.sphere_in_box(args.tris), label="C5 %s 2^24 coherent primaries + incoherent bounces per step")
    if name == args.config:
        if args.width:
            c["W"] = args.width
        if args.height:
            c["H"] = args.height
        if args.bounces >= 0:
            c["bounces"] = args.bounces
        if args.cpu_step:
            c["cpu_step"] = args.cpu_step
    c["name"] = name
    return c


def workload_name(cfg, sc):
    lab = cfg["label"]
    n = lab.count("%")
    if n == 1:
        return lab % sc.name
    return lab % (sc.name, cfg["W"], cfg["H"], cfg["bounces"] + 2, cfg["bounces"])


def config_dict(cfg, sc, world):
    """Identical in the b200 and the reference arm."""
    return {"workload": workload_name(cfg, sc), "triangles": int(sc.n_triangles()),
            "parallelism": "replicated scene, samples mod %d, one NCCL reduce per pass" % world,
            "l2": "per-step path state + queues (%.0f MB) exceed the 126 MB L2; no explicit flush" % (cfg["W"] * cfg["H"] * cfg["spp"] * 468 / 1e6),   # per path: 17 state planes x 16 B + seed 8 + 4 queues x 40 + hit record 20 + visibility 8
            "cpu_sample": "every %d-th pixel in x and y" % cfg["cpu_step"]}


def measured_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/traffic.json); None when absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        return float(t["kernels"][kernel]["dram_bytes_per_launch"]), t.get("source", "")
    except Exception:
        return None, ""


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe).  Started before the warm-up (nvidia-smi
    takes a while to come up); mark_begin()/mark_end() bracket the timed region, only samples inside it are reported."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        time.sleep(0.1)
        self.proc.terminate()
        try:
            text, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            return out
        rows = []
        for line in text.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[1]), float(f[2]), f[5:9]))
            except ValueError:
                continue
        inside = [r for r in rows if self.t0 is not None and self.t1 is not None and self.t0 - 0.02 <= r[0] <= self.t1 + 0.02]
        used, scope = (inside, "timed region") if inside else (rows, "whole run (no sample fell inside the timed region)")
        reasons = set()
        for r in used:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if used:
            out = {"sm_mhz": float(np.median([r[1] for r in used])), "sm_max_mhz": float(max(r[2] for r in used)), "reasons": sorted(reasons),
                   "samples": len(used), "scope": scope}
        return out


# ------------------------------------------------------------------------------------------------ CPU legs (oracle = test infrastructure)
def host_prep(rtdx, sc, W, H):
    """The host-side data preparation of the reference's Renderer slices (librdx_prep.so: no engine, no CUDA inside)."""
    props, descs = rtdx.instance_properties([i[1] for i in sc.instances], [i[0] for i in sc.instances])
    lights = rtdx.collect_emissive_triangles(sc)
    cam = rtdx.camera_params(sc.eye, sc.center, sc.up, W / H)
    return props, descs, lights, cam


def cpu_oracle_sample(cfg, n_threads, cam, osc, first_sample=0):
    """The CPU port on every cpu_step-th pixel of one step of the workload.  Returns (Mrays/s, rays, seconds, image)."""
    t0 = time.perf_counter()
    kw = dict(bounces=cfg["bounces"], flags=cfg["flags"], step=cfg["cpu_step"])
    if n_threads <= 1:
        img, ctr = osc.render(cam, cfg["W"], cfg["H"], first_sample, cfg["spp"], **kw)
    else:
        img, ctr = osc.render_threads(cam, cfg["W"], cfg["H"], first_sample, cfg["spp"], n_threads, **kw)
    dt = time.perf_counter() - t0
    rays = ctr["closest_rays"] + ctr["shadow_rays"]
    return rays / dt / 1e6, rays, dt, img


def cpu_trace_sample(rtdx, cfg, cam, osc, n_threads):
    """C5 on the CPU: the oracle's ray caster on a bounded subset of the coherent batch."""
    import threading
    rays = rtdx.scenes.camera_rays(cam, cfg["W"], cfg["H"], step=cfg["cpu_step"])
    bounds = np.linspace(0, rays.size, n_threads + 1).astype(np.int64)
    parts = [None] * n_threads

    def work(i):
        parts[i] = osc.trace(rays[bounds[i]:bounds[i + 1]])
    t0 = time.perf_counter()
    ts = [threading.Thread(target=work, args=(i,)) for i in range(n_threads)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    dt = time.perf_counter() - t0
    return rays.size / dt / 1e6, rays.size, dt, (rays, np.concatenate(parts))


def oracle_trace_threads(osc, rays, n_threads):
    """osc.trace over the host threads (ctypes releases the GIL; the oracle scene is read-only while tracing)."""
    import threading
    rays = np.ascontiguousarray(rays)
    bounds = np.linspace(0, rays.size, n_threads + 1).astype(np.int64)
    parts = [None] * n_threads

    def work(i):
        parts[i] = osc.trace(rays[bounds[i]:bounds[i + 1]])
    ts = [threading.Thread(target=work, args=(i,)) for i in range(n_threads)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    return np.concatenate(parts)


def crc_of(img, step):
    return int(zlib.crc32(np.ascontiguousarray(img[::step, ::step]).tobytes()))


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (the reference is Windows/DX12-only),
    on all host threads, a bounded sample of the workload per step.  Loads no engine library."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import rtdx
    from oracle import orc
    cfg = config_of(args.config, args)
    sc = cfg["scene"](rtdx)
    props, descs, lights, cam = host_prep(rtdx, sc, cfg["W"], cfg["H"])
    osc = orc.OracleScene(sc, props, lights)           # BVH2 build is not timed (the GPU's BLAS build is not either)
    cores = os.cpu_count() or 1
    rays_tot, t_tot, img0 = 0, 0.0, None
    for k in range(args.warmup + args.steps):
        if cfg["kind"] == "trace":
            _, rays, dt, res = cpu_trace_sample(rtdx, cfg, cam, osc, cores)
        else:
            _, rays, dt, res = cpu_oracle_sample(cfg, cores, cam, osc, first_sample=k * cfg["spp"])
            if k == 0:
                img0 = res
        if k >= args.warmup:
            rays_tot += rays; t_tot += dt
    val = rays_tot / t_tot / 1e6
    sample = "every %d-th pixel in x and y of %dx%d, %d spp, per step (%d rays/step)" % (cfg["cpu_step"], cfg["W"], cfg["H"], cfg["spp"], rays_tot // max(args.steps, 1))
    parity = None
    if img0 is not None:       # the b200 arm prints the CRC of ITS accumulation of the same pixels of sample 0: equal CRCs = bit-identical images
        parity = {"pixels": int(img0[::cfg["cpu_step"], ::cfg["cpu_step"]].shape[0] * img0[::cfg["cpu_step"], ::cfg["cpu_step"]].shape[1]),
                  "crc32_accum_subsample": crc_of(img0, cfg["cpu_step"]), "sample": 0}
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * t_tot / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_dict(cfg, sc, args.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "parity": parity,
        "engine_library_loaded": rtdx._lib is not None,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------ GPU legs
class Dist:
    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0")); self.world = int(os.environ.get("WORLD_SIZE", "1")); self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device — the engine has no CPU fallback")
        torch.cuda.set_device(self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.stream = torch.cuda.Stream()        # a real (non-default) stream: the engine and the events use it
        torch.cuda.set_stream(self.stream)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_sum(self, values):
        t = self.torch.tensor(values, device="cuda", dtype=self.torch.float64)
        if self.world == 1:
            return list(values), list(values)
        a = t.clone(); self.dist.all_reduce(a, op=self.dist.ReduceOp.MAX)
        b = t.clone(); self.dist.all_reduce(b, op=self.dist.ReduceOp.SUM)
        return a.tolist(), b.tolist()


def warm_build_ms(rtdx, D, sc):
    """BLAS build times of a SECOND upload of the scene's models (a fresh context): the first build of a process also pays for the lazy
    loading of the builder's kernels and cub's first-use set-up (10 K triangles and 50 M read alike then), which is not the build."""
    ctx = rtdx.Context(64, 64, device=D.local, stream=D.stream.cuda_stream)
    ids = [ctx.upload_model(m["vertices"], m["indices"], m["material_id_offset"]) for m in sc.models]
    out = [ctx.blas_info(i)["build_ms"] for i in ids]
    ctx.close()
    return out


def make_context(rtdx, D, cfg, sc):
    ctx = rtdx.Context(cfg["W"], cfg["H"], bounces=cfg["bounces"], flags=cfg["flags"], samples_per_pass=cfg["spp"], device=D.local,
                       stream=D.stream.cuda_stream)
    up = ctx.upload_scene(sc)
    if D.world > 1:
        rtdx.dist.init_engine_comm(ctx, D.rank, D.world)
    return ctx, up


def traversal_stats(rtdx, ctx, cfg, rank):
    """Per-ray traversal statistics for the roofline (instrumented kernel variant, untimed, same rays as a timed pass)."""
    spp = cfg["spp"]
    ctx.render_pass(rank * spp, spp); ctx.synchronize()
    ctx.reset_counters(); ctx.set_option(rtdx.OPT_TRACE_STATS, 1)
    ctx.reset_accum(); ctx.render_pass(rank * spp, spp); ctx.synchronize()
    st = ctx.counters(); ctx.set_option(rtdx.OPT_TRACE_STATS, 0)
    n = max(st["closest_rays"], 1)
    n_node, n_tri, n_inst = st["nodes_visited"] / n, st["tris_tested"] / n, st["instances_entered"] / n
    return n_node, n_tri, n_inst, 32 + 20 + 80 * n_node + 48 * n_tri + 64 * n_inst          # SURVEY.md §8d


def roofline_of(rtdx, ctx, cfg, steps, first, rank, world, stats, blas):
    """The same steps again with CUDA events around every traversal launch: achieved = algorithmic bytes / traversal time."""
    n_node, n_tri, n_inst, b_ray = stats
    spp = cfg["spp"]
    ctx.set_option(rtdx.OPT_STAGE_TIMING, 1)
    ctx.reset_counters()
    trace_ms, pass_ms = 0.0, 0.0
    for k in range(steps):
        ctx.render_pass((first + k) * world * spp + rank * spp, spp)
        tr, tot = ctx.last_pass_ms()
        trace_ms += tr; pass_ms += tot
    c = ctx.counters()
    ctx.set_option(rtdx.OPT_STAGE_TIMING, 0)
    peak, peak_src = peaks()
    n_launch = (cfg["bounces"] + 3) * steps
    achieved = (c["closest_rays"] * b_ray) / (trace_ms * 1e-3) / 1e9 if trace_ms > 0 else 0.0
    traffic, traffic_src = measured_traffic("trace_kernel<closest>") if cfg["name"] == "C2" else (None, "")
    return {"bound": "hbm", "kernel": "trace_kernel<closest>", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": ("ncu --set full, dram read+write bytes per launch (profiles/traffic.json <- %s)" % traffic_src) if traffic else None,
            "algorithmic_bytes_per_launch": c["closest_rays"] * b_ray / n_launch, "peak_source": peak_src, "bytes_per_ray": b_ray,
            "nodes_per_ray": n_node, "tris_per_ray": n_tri, "instances_per_ray": n_inst, "launches": n_launch,
            "avg_launch_ms": trace_ms / n_launch, "rays_per_launch": c["closest_rays"] / n_launch,
            "trace_share_of_step": trace_ms / pass_ms if pass_ms else None,
            "note": "BVH %.1f MB (L2-resident below ~100 MB: HBM peak is then the conservative denominator, SURVEY.md §8d); instance entries count every "
                    "64-B record read, incl. those rejected by the object-space bounds; per-launch durations from the same steps re-run with CUDA "
                    "events around every traversal launch (one path range per pass, one pass at a time, full-size launches); the timed steps of "
                    "`value` are consecutive passes, which the engine overlaps two at a time (RTX_OPT_PASS_PIPELINE), the steps of `e2e` "
                    "(instances + camera + pass + read-back per frame) run one at a time as 2 concurrent path ranges" % (sum(b["bytes"] for b in blas) / 1e6)}


def parity_of(rtdx, ctx, cfg, up, sc, osc, img, cores):
    """Bit-compares the oracle image of the cpu_baseline sample (sample 0, every cpu_step-th pixel) with the GPU accumulation of the same
    sample, and the hit ids of the primary rays of those pixels."""
    step, spp = cfg["cpu_step"], cfg["spp"]
    ctx.reset_accum(); ctx.render_pass(0, spp); ctx.synchronize()
    gpu = ctx.read_accum()
    a, b = gpu[::step, ::step], img[::step, ::step]
    fm = int((a.view(np.uint32) != b.view(np.uint32)).sum())
    rays = rtdx.scenes.camera_rays(up["camera"], cfg["W"], cfg["H"], step=step)
    g, r = ctx.trace(rays), oracle_trace_threads(osc, rays, n_threads=cores)
    hit = r["inst"] != 0xFFFFFFFF
    hm = int((g["inst"] != r["inst"]).sum() + (g["prim"][hit] != r["prim"][hit]).sum())
    return {"pixels": int(a.shape[0] * a.shape[1]), "floats": int(a.size), "float_mismatches": fm, "rays": int(rays.size), "hit_id_mismatches": hm,
            "t_u_v_mismatches": int(sum((g[k][hit].view(np.uint32) != r[k][hit].view(np.uint32)).sum() for k in ("t", "u", "v"))),
            "crc32_accum_subsample": crc_of(gpu, step), "sample": 0, "tolerance": 0,
            "against": "oracle/ (CPU port of the reference's shaders, pinned to their text: tests/test_ref_pins.py)"}


def fast_math_leg(rtdx, D, cfg, sc, ctx_exact, steps, warmup):
    """The opt-in RTX_FLAG_FAST_MATH mode (shading stages with FMA contraction and approximate div / sqrt / rsqrt): throughput of the same
    steps and the distance of its image from the exact (parity) mode over the same 16 samples.  Reported beside the headline, never as it."""
    torch = D.torch
    spp = cfg["spp"]
    ctx = rtdx.Context(cfg["W"], cfg["H"], bounces=cfg["bounces"], flags=cfg["flags"] | rtdx.FLAG_FAST_MATH, samples_per_pass=spp, device=D.local,
                       stream=D.stream.cuda_stream)
    ctx.upload_scene(sc)
    for k in range(warmup):
        ctx.render_pass(k * spp, spp)
    D.barrier(); ctx.reset_counters()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(steps):
        ctx.render_pass((warmup + k) * spp, spp)
    e1.record(); D.barrier()
    ms = e0.elapsed_time(e1)
    c = ctx.counters()
    imgs = []
    for cx in (ctx_exact, ctx):
        cx.reset_accum()
        for k in range(16):
            cx.render_pass(k * spp, spp)
        cx.synchronize()
        a = cx.read_accum().astype(np.float64)
        imgs.append(a[..., :3] / np.maximum(a[..., 3:4], 1))
    ctx.close()
    mean = imgs[0].mean()
    le, lf = imgs[0].mean(-1), imgs[1].mean(-1)
    rel = np.abs(le - lf) / np.maximum(le, 1e-3 * mean)
    return {"value": (c["closest_rays"] + c["shadow_rays"]) / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms / max(steps, 1),
            "mean_image_rel_diff": float(abs(imgs[1].mean() - mean) / mean), "rel_rmse_16spp": float(np.sqrt(((imgs[0] - imgs[1]) ** 2).mean()) / mean),
            "pixels_bit_identical_frac_16spp": float((imgs[0] == imgs[1]).all(-1).mean()), "median_pixel_rel_diff_16spp": float(np.median(rel)),
            "pixels_more_than_20pct_apart_frac_16spp": float((rel > 0.2).mean()),
            "note": "opt-in RTX_FLAG_FAST_MATH; not bit-identical to the oracle (paths diverge at discrete decisions, so at 16 spp the RMSE is "
                    "that of the few diverged fireflies); tolerance stated and tested at 256 spp in tests/test_gpu_parity.py::test_fast_math_mode_converges_to_the_exact_image"}


def run_render(rtdx, D, cfg, args, steps, warmup, full):
    """One render config on this rank's GPU.  full = also e2e, clocks, roofline; returns the JSON-ready dict (rank 0) or None."""
    torch = D.torch
    rank, world = D.rank, D.world
    clocks = ClockSampler(D.local) if full else None
    if clocks:
        clocks.start()                       # long before the timed region: nvidia-smi needs time to come up
    sc = cfg["scene"](rtdx)
    W, H, spp = cfg["W"], cfg["H"], cfg["spp"]
    ctx, up = make_context(rtdx, D, cfg, sc)
    blas = [ctx.blas_info(i) for i in up["model_ids"]]
    if full:
        for b, w in zip(blas, warm_build_ms(rtdx, D, sc)):
            b["build_ms_warm"] = w
    stats = traversal_stats(rtdx, ctx, cfg, rank)

    def step_resident(k):
        ctx.render_pass(k * world * spp + rank * spp, spp)
        if world > 1:
            ctx.reduce_accum()               # one NCCL reduce of gPermanentData per progressive pass, on the engine's side stream

    ctx.reset_accum()
    for k in range(warmup):
        step_resident(k)
    D.barrier(); ctx.reset_counters()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if clocks:
        clocks.mark_begin()
    e0.record()
    for k in range(steps):
        step_resident(warmup + k)
    e1.record()
    D.barrier()                              # (synchronises the device: the last reduce on the side stream is complete as well)
    if clocks:
        clocks.mark_end()
    ms = e0.elapsed_time(e1)
    clk = clocks.stop() if clocks else None
    cnt = ctx.counters()
    if full and args.dump_outputs and rank == 0:
        # gPermanentData after the last timed pass (the sum of the warm-up and timed samples; with N ranks, the reduced sum) and the
        # ray / path counts of the timed steps, before the roofline and e2e legs render into the same context
        accum = ctx.read_accum().reshape(-1, 4)
        out = {"counters": [cnt["closest_rays"], cnt["shadow_rays"], cnt["paths"]]}
        if accum.shape[0] > DUMP_SAMPLE_PIXELS:
            out["accum_rows"] = seeded_rows(accum.shape[0], DUMP_SAMPLE_PIXELS)
            out["accum"] = accum[out["accum_rows"]]
        else:
            out["accum"] = accum.reshape(H, W, 4)
        dump_outputs(args.dump_outputs, out)
    rays = cnt["closest_rays"] + cnt["shadow_rays"]
    mx, sm = D.max_sum([ms, float(rays), float(cnt["kernel_launches"])])
    ms, rays_all, launches = mx[0], sm[1], int(sm[2])
    res = {"value": rays_all / (ms * 1e-3) / 1e6, "ms_per_step": ms / max(steps, 1), "gpu_launches": launches,
           "rays_per_path": rays / max(cnt["paths"], 1), "blas": blas, "clocks": clk}
    res["roofline"] = roofline_of(rtdx, ctx, cfg, steps if full else min(steps, 4), warmup, rank, world, stats, blas)

    if full:
        # ---- end to end through the C ABI with host buffers (TLAS refit + camera upload + render (+ reduce) + RGBA8 read-back per step)
        pins = []

        def pinned_copy(a):                  # the step's inputs live in pinned host memory
            t = torch.empty(a.nbytes, dtype=torch.uint8, pin_memory=True)
            pins.append(t)
            n = t.numpy()
            n[:] = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
            return n.view(a.dtype).reshape(a.shape)
        props, descs, cam = pinned_copy(up["props"]), pinned_copy(up["descs"]), pinned_copy(up["camera"])
        h2d = int(props.nbytes + descs.nbytes + cam.nbytes); d2h = W * H * 4
        ctx.reset_accum()
        # the frame's read-back targets (pinned host memory): one frame is kept in flight, so the RGBA8 copy of frame k overlaps the
        # rendering of frame k+1 (rtx_read_output_async / rtx_wait_output); every frame's image is complete on the host before the timed
        # region ends.  With N ranks the image is rank 0's (it resolves the reduced sum).
        out_pinned = [torch.empty((H, W, 4), dtype=torch.uint8, pin_memory=True).numpy() for _ in range(2)]

        def step_e2e(k):
            ctx.set_instances(descs, props)
            ctx.set_camera(cam)
            ctx.render_pass(k * world * spp + rank * spp, spp)
            if world > 1:
                ctx.reduce_accum()
            if rank == 0:
                ctx.wait_output()            # frame k-1's image is on the host (the consumer may use it now)
                ctx.read_output_async(out_pinned[k & 1])

        for k in range(min(warmup, 2)):
            step_e2e(k)
        ctx.wait_output()
        D.barrier(); ctx.reset_counters()
        e0.record()
        t0 = time.perf_counter()
        for k in range(steps):
            step_e2e(warmup + k)
        ctx.wait_output()
        e1.record()
        D.barrier()
        e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
        c2 = ctx.counters()
        mx, sm = D.max_sum([e2e_ms, float(c2["closest_rays"] + c2["shadow_rays"])])
        res["e2e"] = {"value": sm[1] / (mx[0] * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                      "ms_per_step": mx[0] / max(steps, 1)}

    if full and world == 1 and not args.no_extras:
        res["fast_math"] = fast_math_leg(rtdx, D, cfg, sc, ctx, steps, warmup)

    # ---- CPU leg on rank 0: the oracle on a bounded sample (timed, single thread), its image bit-compared with the GPU's
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import orc
        cores = os.cpu_count() or 1
        osc = orc.OracleScene(sc, up["props"], up["lights"])
        threads = 1 if full else cores       # the headline config reports the single-thread port; the compact runs only need the image
        v, r, dt, img = cpu_oracle_sample(cfg, threads, up["camera"], osc)
        res["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                               "sample": "every %d-th pixel in x and y of %dx%d, %d spp (%d rays in %.1f s, %d thread(s), host has %d cores)" % (
                                   cfg["cpu_step"], W, H, spp, r, dt, threads, cores)}
        res["parity"] = parity_of(rtdx, ctx, cfg, up, sc, osc, img, cores)
    res["config"] = config_dict(cfg, sc, world)
    D.barrier()
    ctx.close()
    return res


def run_trace(rtdx, D, cfg, args, steps, warmup):
    """C5: raw TraceRay batches (rtx_trace_device): 2^24 coherent primaries and the incoherent bounces from their hits."""
    torch = D.torch
    sc = cfg["scene"](rtdx)
    ctx = rtdx.Context(64, 64, device=D.local, stream=D.stream.cuda_stream)
    up = ctx.upload_scene(sc)
    blas = [ctx.blas_info(i) for i in up["model_ids"]]
    for b, w in zip(blas, warm_build_ms(rtdx, D, sc)):
        b["build_ms_warm"] = w
    cam = rtdx.camera_params(sc.eye, sc.center, sc.up, 1.0)
    prim = rtdx.scenes.camera_rays(cam, cfg["W"], cfg["H"])
    rays = torch.from_numpy(prim.view(np.float32).reshape(-1, 8)).cuda()
    n = rays.shape[0]
    hits = torch.empty((n, 5), dtype=torch.float32, device="cuda")
    ctx.trace_device(rays.data_ptr(), n, hits.data_ptr()); torch.cuda.synchronize()
    gen = torch.Generator(device="cuda"); gen.manual_seed(7)
    t = hits[:, 0:1]
    o = rays[:, 0:3] + rays[:, 4:7] * t
    d = torch.randn((n, 3), device="cuda", generator=gen); d = d / d.norm(dim=1, keepdim=True)
    inc = torch.cat([o, torch.full((n, 1), 1e-3, device="cuda"), d, torch.full((n, 1), 1e4, device="cuda")], dim=1)
    inc = inc[hits[:, 4].view(torch.int32) != -1].contiguous()
    peak, peak_src = peaks()
    out = {}
    for name, r in (("coherent", rays), ("incoherent", inc)):
        m = r.shape[0]
        h = torch.empty((m, 5), dtype=torch.float32, device="cuda")
        ctx.reset_counters()
        ctx.trace_device(r.data_ptr(), m, h.data_ptr(), stats=True); torch.cuda.synchronize()
        st = ctx.counters()
        b_ray = 52 + (80 * st["nodes_visited"] + 48 * st["tris_tested"] + 64 * st["instances_entered"]) / m
        for _ in range(warmup):
            ctx.trace_device(r.data_ptr(), m, h.data_ptr())
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            ctx.trace_device(r.data_ptr(), m, h.data_ptr())
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        if args.dump_outputs and D.rank == 0:
            keep = seeded_rows(m, DUMP_SAMPLE_RAYS)
            dump_outputs(args.dump_outputs, {"hits_" + name: hit_records(h[torch.from_numpy(keep).cuda()].cpu().numpy()),
                                             "hits_%s_rows" % name: keep})
        out[name] = {"rays": int(m), "ms_per_batch": ms, "value": m / ms / 1e3, "bytes_per_ray": b_ray, "achieved_gbs": m * b_ray / ms / 1e6,
                     "frac": m * b_ray / ms / 1e6 / peak, "nodes_per_ray": st["nodes_visited"] / m, "tris_per_ray": st["tris_tested"] / m}
    total_rays = out["coherent"]["rays"] + out["incoherent"]["rays"]
    total_ms = out["coherent"]["ms_per_batch"] + out["incoherent"]["ms_per_batch"]
    res = {"value": total_rays / total_ms / 1e3, "ms_per_step": total_ms, "gpu_launches": 3 * 2 * steps, "batches": out, "blas": blas,
           "roofline": {"bound": "hbm", "kernel": "trace_kernel<closest>", "achieved": out["incoherent"]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                        "frac": out["incoherent"]["frac"], "traffic": None, "peak_source": peak_src, "batch": "incoherent",
                        "note": "includes the split / pack kernels of rtx_trace_device (3 launches per batch)"}}
    if D.rank == 0 and not args.no_cpu_baseline:
        from oracle import orc
        cores = os.cpu_count() or 1
        osc = orc.OracleScene(sc, up["props"], up["lights"])
        v, nr, dt, (sub, ref) = cpu_trace_sample(rtdx, cfg, cam, osc, cores)
        res["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                               "sample": "every %d-th primary ray in x and y of the coherent batch (%d rays in %.1f s)" % (cfg["cpu_step"], nr, dt)}
        isub = inc[:1 << 16].cpu().numpy().view(rtdx.ray_dt).reshape(-1)
        allr = np.concatenate([sub, isub])
        refa = np.concatenate([ref, oracle_trace_threads(osc, isub, n_threads=cores)])
        g = ctx.trace(allr)
        hit = refa["inst"] != 0xFFFFFFFF
        res["parity"] = {"rays": int(allr.size), "hit_id_mismatches": int((g["inst"] != refa["inst"]).sum() + (g["prim"][hit] != refa["prim"][hit]).sum()),
                         "t_u_v_mismatches": int(sum((g[k][hit].view(np.uint32) != refa[k][hit].view(np.uint32)).sum() for k in ("t", "u", "v"))),
                         "tolerance": 0, "against": "oracle/ BVH2 ray caster"}
    res["config"] = config_dict(cfg, sc, D.world)
    ctx.close()
    return res


def run_c4_strong(rtdx, D, args):
    """BASELINE config C4: 3840x2160 progressive render of the C2 scene, S samples per pixel per step split over the N ranks
    (rank r renders samples s = r (mod N)), one NCCL reduce of the 133 MB accumulation buffer per pass.  STRONG scaling: the work of a
    step is fixed, the time should fall as 1/N."""
    torch = D.torch
    S = max(args.c4_spp, D.world)
    cfg = dict(kind="render", W=3840, H=2160, bounces=6, flags=0, spp=1, cpu_step=16, name="C4",
               scene=lambda r: r.scenes.mesh_room(n=args.side, seed=1), label="C4 %s %dx%d progressive, depth %d (bounces=%d)")
    sc = cfg["scene"](rtdx)
    ctx, up = make_context(rtdx, D, cfg, sc)
    mine = list(range(D.rank, S, D.world))

    def step(k):
        for s in mine:
            ctx.render_pass(k * S + s, 1)
            if D.world > 1:
                ctx.reduce_accum()
    step(0)
    D.barrier(); ctx.reset_counters()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = 3
    e0.record()
    for k in range(steps):
        step(1 + k)
    e1.record()
    D.barrier()
    c = ctx.counters()
    mx, sm = D.max_sum([e0.elapsed_time(e1), float(c["closest_rays"] + c["shadow_rays"]), float(c["kernel_launches"])])
    ctx.close()
    return {"workload": workload_name(cfg, sc) + ", %d spp per step over %d GPU(s)" % (S, D.world), "scaling": "strong", "value": sm[1] / (mx[0] * 1e-3) / 1e6,
            "unit": UNIT, "ms_per_step": mx[0] / steps, "spp_per_step": S, "steps": steps, "gpu_launches": int(sm[2])}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    import rtdx
    import importlib
    rtdx.dist = importlib.import_module("royaltracer-dx_b200.dist")
    D = Dist()
    cfg = config_of(args.config, args)
    if cfg["kind"] == "trace":
        res = run_trace(rtdx, D, cfg, args, args.steps, args.warmup)
    else:
        res = run_render(rtdx, D, cfg, args, args.steps, args.warmup, full=True)
    extras, c4 = {}, None
    if not args.no_extras and args.config == "C2":
        if D.world == 1:                     # compact runs of the other BASELINE configs, so that the driver's record carries them
            for name in ("C1", "C3"):
                r = run_render(rtdx, D, config_of(name, args), args, 8, 3, full=False)
                extras[name] = {k: r.get(k) for k in ("config", "value", "ms_per_step", "rays_per_path", "roofline", "cpu_baseline", "parity")}
            for tris in (1_000_000, 10_000_000):
                a2 = argparse.Namespace(**vars(args)); a2.tris = tris; a2.no_cpu_baseline = args.no_cpu_baseline or tris > 2_000_000
                a2.dump_outputs = ""
                r = run_trace(rtdx, D, config_of("C5", a2), a2, 5, 2)
                extras["C5_%dM" % (tris // 1_000_000)] = {k: r.get(k) for k in ("config", "value", "ms_per_step", "batches", "roofline", "cpu_baseline", "parity", "blas")}
        c4 = run_c4_strong(rtdx, D, args)
    if D.rank == 0:
        line = {
            "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": D.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": res["config"], "rays_per_path": res.get("rays_per_path"),
            "e2e": res.get("e2e"), "gpu_launches": res["gpu_launches"], "clocks": res.get("clocks"), "roofline": res["roofline"],
            "cpu_baseline": res.get("cpu_baseline"), "parity": res.get("parity"), "blas": res.get("blas"),
        }
        if res.get("fast_math"):
            line["fast_math"] = res["fast_math"]
        if "batches" in res:
            line["batches"] = res["batches"]
        if extras:
            line["configs"] = extras
        if c4:
            line["c4_strong"] = c4
        print(json.dumps(line), flush=True)
    if D.world > 1:
        D.dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
