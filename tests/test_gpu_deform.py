"""-m gpu: deforming meshes (rtx_update_model / rtx_update_model_device, DXR PERFORM_UPDATE).  After every update the engine's hits,
ray counts, reservoirs and accumulation equal the oracle's over the deformed vertices bit for bit (tolerance 0, as in test_gpu_parity.py),
whether the BLAS was refitted, rebuilt, or uploaded fresh."""
import numpy as np
import pytest

from deform_util import oracle_update, small_model_scene, with_vertices
from util import bits, compare_hits, host_inputs, random_rays

pytestmark = pytest.mark.gpu

AMPLITUDES = (0.1, 0.25, 0.5, 1.0)      # a sequence of growing deformations


def _assert_hits_equal(gpu, ref, tag=""):
    r = compare_hits(gpu, ref)
    assert r["inst"] == 0 and r["prim"] == 0 and r["t"] == 0 and r["u"] == 0 and r["v"] == 0, (tag, r)


def _assert_same_hits(a, b, tag=""):
    for k in ("inst", "prim", "t", "u", "v"):
        assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), (tag, k)


def _rays(rtdx, cam, W, H, lo, hi, n, seed):
    rng = np.random.RandomState(seed)
    return np.concatenate([rtdx.scenes.camera_rays(cam, W, H), random_rays(rtdx, rng, n, lo, hi)])


def _blobs(rtdx, lattice):
    """instanced_blobs with ONE blob model instanced lattice^3 times (model 0) plus its emissive twin (model 1)."""
    return rtdx.scenes.instanced_blobs(n_models=1, n_side=6, lattice=lattice, emissive_fraction=0.1)


@pytest.mark.parametrize("scene_name", ["mesh_room_40", "single_node", "blobs_refit_tlas", "blobs_one_node_tlas"])
def test_refit_hits_equal_brute_force_rebuild_and_fresh_upload(rtdx, orc, scene_name):
    sc, lo, hi = {"mesh_room_40": lambda: (rtdx.scenes.mesh_room(n=40), (-5, 0.1, -5), (5, 5.9, 5)),
                  "single_node": lambda: (small_model_scene(rtdx), (-2.5, 0.1, -2.5), (2.5, 2.9, 2.5)),
                  "blobs_refit_tlas": lambda: (_blobs(rtdx, 4), -2.5, 2.5),           # 64 instances: a refitted multi-node TLAS
                  "blobs_one_node_tlas": lambda: (_blobs(rtdx, 2), -1.5, 1.5)}[scene_name]()   # 8 instances: the one-node TLAS
    W, H = 96, 64
    refit = rtdx.Context(W, H); up = refit.upload_scene(sc)
    rebuild = rtdx.Context(W, H); rebuild.upload_scene(sc)
    nodes = refit.blas_info(0)["n_nodes"]
    assert scene_name != "single_node" or nodes == 1
    assert scene_name != "mesh_room_40" or nodes > 100
    rays = _rays(rtdx, up["camera"], W, H, lo, hi, 30000, 17)
    base = sc.models[0]["vertices"]
    for k, amp in enumerate(AMPLITUDES):
        v = rtdx.scenes.deform(base, 0.2 * k, amp, seed=9)
        refit.update_model(0, v)
        rebuild.update_model(0, v, mode=rtdx.UPDATE_REBUILD)
        g = refit.trace(rays)
        _, osc, _ = oracle_update(orc, sc, up["props"], 0, v, lights=up["lights"])
        _assert_hits_equal(g, osc.trace(rays, mode=1), (scene_name, amp, "oracle BVH2"))
        sub = rays[::17]
        _assert_hits_equal(g[::17], osc.trace(sub, mode=0), (scene_name, amp, "brute force"))
        _assert_same_hits(g, rebuild.trace(rays), (scene_name, amp, "rebuild"))
        fresh = rtdx.Context(W, H); fresh.upload_scene(with_vertices(sc, 0, v))
        _assert_same_hits(g, fresh.trace(rays), (scene_name, amp, "fresh upload"))
        fresh.close()
        assert (g["inst"] != rtdx.MISS).mean() > 0.05
        assert refit.blas_info(0)["n_nodes"] == nodes                       # a refit keeps the topology
    refit.close(); rebuild.close()


def test_bounds_that_leave_the_old_box(rtdx, orc):
    """Scaled x4 and moved out of its old bounds, flattened to a plane, collapsed to one point: stale object-space rejection bounds or
    a stale padding would cull or miss hits."""
    for sc in (rtdx.scenes.mesh_room(n=8), small_model_scene(rtdx)):
        W, H = 64, 48
        ctx = rtdx.Context(W, H); up = ctx.upload_scene(sc)
        base = sc.models[0]["vertices"]
        big = base.copy(); big["position"] = base["position"] * np.float32(4.0) + np.array([9.0, 1.0, -7.0], dtype=np.float32)
        flat = base.copy(); flat["position"][:, 1] = np.float32(1.25)
        point = base.copy(); point["position"][:] = np.array([0.5, 1.0, 0.25], dtype=np.float32)
        rays = _rays(rtdx, up["camera"], W, H, (-12, -4, -12), (16, 8, 12), 20000, 23)
        for tag, v in (("x4 and moved", big), ("flat", flat), ("one point", point), ("back", base)):
            for mode in (rtdx.UPDATE_REFIT, rtdx.UPDATE_REBUILD):
                ctx.update_model(0, v, mode=mode)
                _, osc, _ = oracle_update(orc, sc, up["props"], 0, v, lights=up["lights"])
                _assert_hits_equal(ctx.trace(rays), osc.trace(rays, mode=0), (sc.name, tag, mode))
        ctx.close()


def test_host_bounds_stay_current_for_table_rebuilds(rtdx, orc):
    """A refit through rtx_update_model_device leaves the new bounds on the device; uploading another model then makes
    rtx_set_instances rebuild every per-model table from the host copies, which must hold the refitted bounds."""
    import torch
    sc = rtdx.scenes.mesh_room(n=16)
    W, H = 64, 48
    ctx = rtdx.Context(W, H); up = ctx.upload_scene(sc)
    v = sc.models[0]["vertices"].copy()
    v["position"] = v["position"] * np.float32(1.8) + np.array([1.5, 0.4, -1.0], dtype=np.float32)     # leaves the old box
    t = torch.from_numpy(v.view(np.uint8).copy()).cuda()
    torch.cuda.synchronize()
    ctx.update_model_device(0, t, v.size)
    extra = small_model_scene(rtdx)
    em = extra.models[0]
    mid = ctx.upload_model(em["vertices"], em["indices"], 0)
    xm = np.eye(4); xm[:3, 3] = (-3.5, 0.5, 2.0)
    xms = [i[1] for i in sc.instances] + [rtdx.xmmatrix_from_colvec(xm)]
    props, descs = rtdx.instance_properties(xms, [0, 1, mid])
    ctx.set_instances(descs, props)
    sc2 = with_vertices(sc, 0, v)
    sc2.models.append({"vertices": em["vertices"], "indices": em["indices"], "material_id_offset": 0})
    sc2.instances = list(sc.instances) + [(2, xms[2])]
    osc = orc.OracleScene(sc2, props, up["lights"])
    rays = _rays(rtdx, up["camera"], W, H, (-5, 0.1, -5), (5, 5.9, 5), 30000, 29)
    _assert_hits_equal(ctx.trace(rays), osc.trace(rays, mode=1))
    ctx.close()


def _render_scene(rtdx):
    sc = rtdx.scenes.mesh_room(n=16)
    v0 = rtdx.scenes.deform(sc.models[0]["vertices"], 0.3, 0.4, seed=1)        # the blob
    v1 = rtdx.scenes.deform(sc.models[1]["vertices"], 0.1, 0.03, seed=2)       # the room with its emitter
    return sc, v0, v1


@pytest.mark.parametrize("flags", [0, 16], ids=["E0", "LEGACY_RR"])
def test_render_across_an_update(rtdx, orc, flags):
    """Two samples on the original meshes, an update of both models (the emissive one with its light list set again), two more
    samples: the accumulation equals the oracle's, which renders the first two samples, updates, and renders the last two into the same
    buffer — with the defaults (pass graph, pipelined passes, two path ranges) and without the pass graph."""
    sc, v0, v1 = _render_scene(rtdx)
    W, H = 384, 192
    bounces = 12 if flags else 3
    props, _, lights, cam = host_inputs(rtdx, sc, W, H)
    osc = orc.OracleScene(sc, props, lights)
    ref = np.zeros((H, W, 4), dtype=np.float32)
    _, c0 = osc.render_threads(cam, W, H, 0, 2, 16, bounces=bounces, flags=flags, accum=ref)
    sc1 = with_vertices(with_vertices(sc, 0, v0), 1, v1)
    lights1 = rtdx.collect_emissive_triangles(sc1)
    assert not np.array_equal(lights1.view(np.uint8), lights.view(np.uint8))
    osc1 = orc.OracleScene(sc1, props, lights1)
    _, c1 = osc1.render_threads(cam, W, H, 2, 2, 16, bounces=bounces, flags=flags, accum=ref)
    for opts in ({}, {rtdx.OPT_PASS_GRAPH: 0}):
        ctx = rtdx.Context(W, H, bounces=bounces, flags=flags)
        ctx.upload_scene(sc)
        for k, val in opts.items():
            ctx.set_option(k, val)
        for s in range(2):
            ctx.render_pass(s, 1)
        ctx.update_model(0, v0)
        ctx.update_model(1, v1)
        ctx.set_emissive_triangles(lights1)
        for s in range(2, 4):
            ctx.render_pass(s, 1)
        ctx.synchronize()
        cnt = ctx.counters()
        assert cnt["closest_rays"] == c0["closest_rays"] + c1["closest_rays"] and cnt["shadow_rays"] == c0["shadow_rays"] + c1["shadow_rays"], opts
        assert (bits(ctx.read_accum()) != bits(ref)).sum() == 0, opts
        ctx.close()


def test_restir_frames_across_updates(rtdx, orc):
    """rtx_render_frame for four frames with the emissive Cornell model deformed between frames (light list set again): reservoirs, ray
    counts and accumulation equal the oracle's frames with the same updates.  Reprojection uses instance matrices only."""
    sc = rtdx.scenes.cornell()
    W, H, bounces = 96, 80, 2
    ctx = rtdx.Context(W, H, bounces=bounces, flags=rtdx.FLAG_RESTIR)
    up = ctx.upload_scene(sc)
    osc = orc.OracleScene(sc, up["props"], up["lights"])
    frames = osc.new_frames(W, H)
    acc = np.zeros((H, W, 4), dtype=np.float32)
    total = [0, 0]
    base = sc.models[0]["vertices"]
    for f in range(4):
        if f:
            v = rtdx.scenes.deform(base, 0.25 * f, 0.05 * f, seed=6)
            ctx.update_model(0, v, mode=rtdx.UPDATE_REFIT if f != 2 else rtdx.UPDATE_REBUILD)
            _, osc2, lights = oracle_update(orc, sc, up["props"], 0, v, rtdx=rtdx)
            ctx.set_emissive_triangles(lights)
            osc.close(); osc = osc2
        ctx.render_frame(f)
        ctx.synchronize()
        octr = osc.render_frame(up["camera"], W, H, f, frames, acc, bounces=bounces, flags=0)
        total[0] += octr["closest_rays"]; total[1] += octr["shadow_rays"]
        cnt = ctx.counters()
        assert (cnt["closest_rays"], cnt["shadow_rays"]) == tuple(total), (f, cnt, total)
        bad = (bits(ctx.read_restir()) != bits(osc.dump_frames(frames, W, H))).any(axis=-1)
        assert bad.sum() == 0, "frame %d: %d pixels with differing reservoirs" % (f, bad.sum())
        assert (bits(ctx.read_accum()) != bits(acc)).sum() == 0, f
    osc.free_frames(frames)
    ctx.close()


def test_device_update_equals_host_update_and_rejects_bad_arguments(rtdx, orc):
    """A torch tensor deformed on the GPU and handed to rtx_update_model_device gives the hits and image of rtx_update_model with the
    same bytes; bad arguments return RTX_ERR_ARG and leave the context usable."""
    import torch
    sc = rtdx.scenes.mesh_room(n=16)
    W, H, bounces = 128, 96, 3
    base = sc.models[0]["vertices"]
    t = torch.from_numpy(base.view(np.float32).reshape(-1, 7).copy()).cuda()
    p = t[:, :3]
    t[:, :3] = p + 0.15 * torch.sin(3.0 * p[:, [1, 2, 0]]) * t[:, 3:6]          # a wave along the normals, computed on the GPU
    torch.cuda.synchronize()
    v = t.cpu().numpy().reshape(-1).view(rtdx.vertex_dt).copy()
    out = []
    for device in (True, False):
        ctx = rtdx.Context(W, H, bounces=bounces)
        up = ctx.upload_scene(sc)
        if device:
            ctx.update_model_device(0, t, base.size)
        else:
            ctx.update_model(0, v)
        ctx.render_pass(0, 2); ctx.synchronize()
        rays = _rays(rtdx, up["camera"], W, H, (-5, 0.1, -5), (5, 5.9, 5), 20000, 31)
        out.append((ctx.trace(rays), ctx.read_accum(), rays))
        if device:
            host = np.ascontiguousarray(v)
            bad = [lambda: ctx.update_model_device(0, t, base.size - 1),                       # wrong count
                   lambda: ctx.update_model_device(7, t, base.size),                           # unknown model
                   lambda: ctx.update_model_device(0, t, base.size, mode=2),                   # unknown mode
                   lambda: ctx.update_model_device(0, host.ctypes.data, base.size),            # host memory
                   lambda: ctx.update_model_device(0, 0, base.size),                           # null
                   lambda: ctx.update_model(0, v[:-1]),
                   lambda: ctx.update_model(0, v, mode=7)]
            for call in bad:
                with pytest.raises(rtdx.RtxError, match="rtx error 1:"):
                    call()
            _assert_same_hits(ctx.trace(rays), out[0][0], "after the rejected calls")
        ctx.close()
    _assert_same_hits(out[0][0], out[1][0])
    assert np.array_equal(bits(out[0][1]), bits(out[1][1]))
    _, osc, _ = oracle_update(orc, sc, up["props"], 0, v, lights=up["lights"])
    _assert_hits_equal(out[0][0], osc.trace(out[0][2], mode=1))


def test_per_frame_deforming_loop_matches_the_unpipelined_loop(rtdx, orc):
    """update_model_device -> set_instances -> set_camera -> render_pass -> read_output_async for six frames: the same images as the
    loop with OPT_PASS_PIPELINE=0 and OPT_FRAME_PIPELINE=0, and the oracle's accumulation."""
    import torch
    sc = rtdx.scenes.mesh_room(n=16)
    W, H, bounces, n_frames = 384, 192, 2, 6
    base = sc.models[0]["vertices"]
    verts = [rtdx.scenes.deform(base, 0.15 * f, 0.3, seed=3) for f in range(n_frames)]
    dev = [torch.from_numpy(v.view(np.uint8).copy()).cuda() for v in verts]
    torch.cuda.synchronize()

    def loop(pipeline):
        ctx = rtdx.Context(W, H, bounces=bounces)
        up = ctx.upload_scene(sc)
        ctx.set_option(rtdx.OPT_PASS_PIPELINE, pipeline); ctx.set_option(rtdx.OPT_FRAME_PIPELINE, pipeline)
        pinned = [torch.empty((H, W, 4), dtype=torch.uint8).pin_memory().numpy() for _ in range(2)]
        images = []
        for f in range(n_frames):
            ctx.update_model_device(0, dev[f], base.size)
            ctx.set_instances(up["descs"], up["props"])
            ctx.set_camera(up["camera"])
            ctx.render_pass(f, 1)
            if f:
                ctx.wait_output(); images.append(pinned[(f - 1) & 1].copy())
            ctx.read_output_async(pinned[f & 1])
        ctx.wait_output(); images.append(pinned[(n_frames - 1) & 1].copy())
        acc = ctx.read_accum()
        ctx.close()
        return images, acc, up

    img_on, acc_on, up = loop(1)
    img_off, acc_off, _ = loop(0)
    assert len(img_on) == n_frames and all(np.array_equal(a, b) for a, b in zip(img_on, img_off))
    assert np.array_equal(bits(acc_on), bits(acc_off))
    ref = np.zeros((H, W, 4), dtype=np.float32)
    for f in range(n_frames):
        _, osc, _ = oracle_update(orc, sc, up["props"], 0, verts[f], lights=up["lights"])
        osc.render_threads(up["camera"], W, H, f, 1, 16, bounces=bounces, flags=0, accum=ref)
        osc.close()
    assert (bits(acc_on) != bits(ref)).sum() == 0
