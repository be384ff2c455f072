"""-m gpu: the light list built on the device (rtx_collect_emissive_triangles).  Its records, their order and their count equal the host
collection rtdx.collect_emissive_triangles over the same state byte for byte, after every kind of update; rendering with it equals the
oracle bit for bit; the per-frame call neither waits nor allocates."""
import os
import time

import numpy as np
import pytest

from deform_util import oracle_update, small_model_scene, with_vertices
from util import bits, host_inputs, load_scene_npz

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
AMPLITUDES = (0.1, 0.25, 0.5, 1.0)      # those of test_gpu_deform.py


def _assert_same_list(got, ref, tag="", nan_aware=False):
    """Byte equality; nan_aware: a NaN field matches any NaN (all-zero-area emitters give 0/0, whose NaN bits differ between the
    host's x86 default NaN and CUDA's canonical one)."""
    assert got.dtype == ref.dtype and got.size == ref.size, (tag, got.size, ref.size)
    g, r = got.view(np.uint32).reshape(-1, 20), ref.view(np.uint32).reshape(-1, 20)
    same = g == r
    if nan_aware:
        same |= np.isnan(g.view(np.float32)) & np.isnan(r.view(np.float32))
    assert same.all(), (tag, int((~same.all(axis=1)).sum()), "records differ")


def _collect_and_check(rtdx, ctx, sc, tag="", nan_aware=False):
    ref = rtdx.collect_emissive_triangles(sc)
    n = ctx.collect_emissive_triangles()
    assert n == ref.size, (tag, n, ref.size)
    _assert_same_list(ctx.read_emissive_triangles(), ref, tag, nan_aware)
    return ref


def _mixed_material_scene(rtdx):
    """small_model_scene with triangles whose face-vertex ids differ (skipped even where one of them is an emitter), an emitter whose Ke
    has a negative component but a positive sum, and a material whose Ke sums to 0."""
    sc = small_model_scene(rtdx)
    extra = np.concatenate([rtdx.scenes.make_material((0, 0, 0), ke=(1.5, -0.5, 0.25)), rtdx.scenes.make_material((0, 0, 0), ke=(1, -1, 0))])
    sc.materials = rtdx.scenes._fill_luts(np.concatenate([sc.materials, extra]))
    POS, ZERO = sc.materials.size - 2, sc.materials.size - 1
    ids = sc.material_ids.copy()
    off1 = sc.models[1]["material_id_offset"]
    ids[off1 + 3 * 12 + 1] = 2                  # the first emitter triangle: mixed
    ids[3 * 1: 3 * 2] = 3                       # tetrahedron triangle 1: the emitter material
    ids[3 * 2: 3 * 3] = (3, 3, 1)               # triangle 2: mixed
    ids[3 * 3: 3 * 4] = POS
    ids[3 * 4: 3 * 5] = ZERO
    sc.material_ids = ids
    return sc


def _no_emitter_scene(rtdx):
    sc = small_model_scene(rtdx)
    sc.materials = sc.materials.copy()
    sc.materials["Ke"][:] = 0
    return sc


SCENES = {
    "cornell": lambda r: r.scenes.cornell(),
    "mesh_room": lambda r: r.scenes.mesh_room(n=40),
    "small_model": small_model_scene,
    "garage_monke": lambda r: load_scene_npz(r, os.path.join(HERE, "golden", "reference_scene.npz")),
    "blobs_ties": lambda r: r.scenes.instanced_blobs(n_models=2, lattice=4, emissive_fraction=0.25),
    "c3_defaults": lambda r: r.scenes.instanced_blobs(),
    "mixed_materials": _mixed_material_scene,
    "no_emitter": _no_emitter_scene,
}


@pytest.mark.parametrize("name", list(SCENES))
def test_same_bytes_as_the_host_collection(rtdx, name):
    sc = SCENES[name](rtdx)
    ctx = rtdx.Context(32, 32)
    up = ctx.upload_scene(sc)
    _assert_same_list(ctx.read_emissive_triangles(), up["lights"], "the list upload_scene set")
    ref = _collect_and_check(rtdx, ctx, sc, name)
    assert name != "c3_defaults" or ref.size == 504600
    assert name != "cornell" or ref.size == 2
    assert name != "no_emitter" or ref.size == 0
    if name == "blobs_ties":        # several instances of one emissive model: equal weights across instances, order decided by the tie rule
        assert np.unique(ref["instanceID"]).size > 1 and np.unique(ref["weight"]).size < ref.size
    _collect_and_check(rtdx, ctx, sc, name + " again")
    ctx.close()


def test_no_emitter_renders_like_an_empty_list(rtdx):
    sc = _no_emitter_scene(rtdx)
    acc = []
    for collect in (True, False):
        ctx = rtdx.Context(48, 32, bounces=2)
        ctx.upload_scene(sc)
        if collect:
            assert ctx.collect_emissive_triangles() == 0
        else:
            ctx.set_emissive_triangles(np.zeros(0, dtype=rtdx.light_dt))
        ctx.render_pass(0, 2)
        acc.append(ctx.read_accum())
        ctx.close()
    assert np.array_equal(bits(acc[0]), bits(acc[1]))


def _tensor(v):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(v).view(np.uint8).copy()).cuda()
    torch.cuda.synchronize()
    return t


@pytest.mark.parametrize("scene_name", ["mesh_room", "blobs"])
def test_after_model_updates(rtdx, scene_name):
    """update_model and update_model_device, refit and rebuild, of the emissive model at growing amplitudes, flattened and collapsed
    to one point (every emitter of zero area: NaN-aware)."""
    if scene_name == "mesh_room":
        sc, m = rtdx.scenes.mesh_room(n=16), 1                   # the room with its emitter quad
    else:
        sc = rtdx.scenes.instanced_blobs(n_models=2, n_side=6, lattice=4, emissive_fraction=0.25)
        m = len(sc.models) - 1                                   # the emissive blob
    base = sc.models[m]["vertices"]
    cases = [("amp %g" % a, rtdx.scenes.deform(base, 0.2 * k, a, seed=9)) for k, a in enumerate(AMPLITUDES)]
    flat = base.copy(); flat["position"][:, 1] = np.float32(1.25)
    point = base.copy(); point["position"][:] = np.array([0.5, 1.0, 0.25], dtype=np.float32)
    cases += [("flat", flat), ("one point", point), ("back", base)]
    ctx = rtdx.Context(32, 32)
    ctx.upload_scene(sc)
    ctx.collect_emissive_triangles()
    for tag, v in cases:
        for device in (False, True):
            for mode in (rtdx.UPDATE_REFIT, rtdx.UPDATE_REBUILD):
                if device:
                    ctx.update_model_device(m, _tensor(v), v.size, mode)
                else:
                    ctx.update_model(m, v, mode)
                _collect_and_check(rtdx, ctx, with_vertices(sc, m, v), (scene_name, tag, device, mode), nan_aware=tag == "one point")
    ctx.close()


def test_after_material_and_instance_changes(rtdx):
    sc = rtdx.scenes.instanced_blobs(n_models=2, n_side=6, lattice=4, emissive_fraction=0.25)
    ctx = rtdx.Context(32, 32)
    up = ctx.upload_scene(sc)
    _collect_and_check(rtdx, ctx, sc, "upload")
    LIGHT = sc.materials.size - 1
    sc2 = with_vertices(sc, 0, sc.models[0]["vertices"])
    for tag, edit in (("light off", lambda k: k.__setitem__(LIGHT, (0, 0, 0))),
                      ("material 1 turned emitter", lambda k: k.__setitem__(1, (0.5, 0.25, 2.0))),
                      ("Ke changed", lambda k: k.__setitem__(LIGHT, (3, 4, 5)))):
        mats = sc2.materials.copy(); edit(mats["Ke"]); sc2.materials = mats
        ctx.set_materials(mats)
        _collect_and_check(rtdx, ctx, sc2, tag)
    ids = sc2.material_ids.copy()
    ids[: 3 * 40] = LIGHT                        # 40 triangles of model 0 become emitters
    ids[3 * 40 + 1] = LIGHT                      # and one mixed triangle
    sc2.material_ids = ids
    ctx.set_material_ids(ids)
    _collect_and_check(rtdx, ctx, sc2, "material ids")
    # other instance lists: half of them (another number of emissive instances), the same models moved, and every emissive one twice
    em = [k for k, (mi, _) in enumerate(sc2.instances) if mi == len(sc2.models) - 1]
    shift = np.float32(0.5) * ((np.arange(16) >= 12) & (np.arange(16) < 15))       # XMMATRIX memory: the translation row
    lists = [sc2.instances[: len(sc2.instances) // 2],
             [(mi, xm + shift) for mi, xm in sc2.instances],
             sc2.instances + [sc2.instances[k] for k in em]]
    for k, inst in enumerate(lists):
        sc3 = with_vertices(sc2, 0, sc2.models[0]["vertices"]); sc3.instances = inst
        props, descs = rtdx.instance_properties([i[1] for i in inst], [up["model_ids"][i[0]] for i in inst])
        ctx.set_instances(descs, props)
        _collect_and_check(rtdx, ctx, sc3, ("instances", k))
    ctx.close()


def test_state_errors_and_launch_count(rtdx):
    sc = small_model_scene(rtdx)
    ctx = rtdx.Context(32, 32)
    with pytest.raises(rtdx.RtxError, match="rtx error 3:"):
        ctx.collect_emissive_triangles()                 # nothing set
    ids = [ctx.upload_model(m["vertices"], m["indices"], m["material_id_offset"]) for m in sc.models]
    props, descs = rtdx.instance_properties([i[1] for i in sc.instances], [ids[i[0]] for i in sc.instances])
    ctx.set_instances(descs, props)
    with pytest.raises(rtdx.RtxError, match="rtx error 3:"):
        ctx.collect_emissive_triangles()                 # no materials
    ctx.set_material_ids(sc.material_ids); ctx.set_materials(sc.materials)
    _collect_and_check(rtdx, ctx, sc, "complete")
    ctx.reset_counters()
    _collect_and_check(rtdx, ctx, sc, "steady")
    assert ctx.counters()["kernel_launches"] == 5
    ctx.upload_model(sc.models[0]["vertices"], sc.models[0]["indices"], 0)
    with pytest.raises(rtdx.RtxError, match="rtx error 3:"):
        ctx.collect_emissive_triangles()                 # the upload invalidated the instance list
    assert ctx.read_emissive_triangles().size == 2       # the list stays what the last collect wrote
    import ctypes as C
    n = C.c_uint32()
    out = np.zeros(1, dtype=rtdx.light_dt)
    assert ctx.lib.rtx_read_emissive_triangles(ctx.handle, out.ctypes.data_as(C.c_void_p), 1, C.byref(n)) == 1 and n.value == 2
    ctx.close()


def _render_scene(rtdx):
    sc = rtdx.scenes.mesh_room(n=16)
    v0 = rtdx.scenes.deform(sc.models[0]["vertices"], 0.3, 0.4, seed=1)        # the blob
    v1 = rtdx.scenes.deform(sc.models[1]["vertices"], 0.1, 0.03, seed=2)       # the room with its emitter
    return sc, v0, v1


@pytest.mark.parametrize("flags", [0, 16], ids=["E0", "LEGACY_RR"])
def test_render_across_an_update(rtdx, orc, flags):
    """test_gpu_deform.py's render across an update with the light list collected on the device: two samples, an update of both
    models, two more samples; accumulation and ray counts equal the oracle's, with and without the pass graph."""
    sc, v0, v1 = _render_scene(rtdx)
    W, H = 384, 192
    bounces = 12 if flags else 3
    props, _, lights, cam = host_inputs(rtdx, sc, W, H)
    osc = orc.OracleScene(sc, props, lights)
    ref = np.zeros((H, W, 4), dtype=np.float32)
    _, c0 = osc.render_threads(cam, W, H, 0, 2, 16, bounces=bounces, flags=flags, accum=ref)
    sc1 = with_vertices(with_vertices(sc, 0, v0), 1, v1)
    lights1 = rtdx.collect_emissive_triangles(sc1)
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
        assert ctx.collect_emissive_triangles() == lights1.size
        for s in range(2, 4):
            ctx.render_pass(s, 1)
        ctx.synchronize()
        cnt = ctx.counters()
        assert cnt["closest_rays"] == c0["closest_rays"] + c1["closest_rays"] and cnt["shadow_rays"] == c0["shadow_rays"] + c1["shadow_rays"], opts
        assert (bits(ctx.read_accum()) != bits(ref)).sum() == 0, opts
        _assert_same_list(ctx.read_emissive_triangles(), lights1)
        ctx.close()


def test_restir_frames_across_updates(rtdx, orc):
    """test_gpu_deform.py's ReSTIR frames with the emissive Cornell model deformed between frames and the light list collected on the
    device: reservoirs, ray counts and accumulation equal the oracle's."""
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
            assert ctx.collect_emissive_triangles() == lights.size
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


def test_per_frame_deforming_emitter_loop(rtdx, orc):
    """update_model_device (the emissive model) -> collect -> set_instances -> set_camera -> render_pass -> read_output_async for six
    frames: the images and accumulation of the same loop with OPT_PASS_PIPELINE=0 and OPT_FRAME_PIPELINE=0, and the oracle's
    accumulation over each frame's host-collected list."""
    import torch
    sc = rtdx.scenes.mesh_room(n=16)
    W, H, bounces, n_frames, m = 384, 192, 2, 6, 1
    base = sc.models[m]["vertices"]
    verts = [rtdx.scenes.deform(base, 0.15 * f, 0.05, seed=3) for f in range(n_frames)]
    dev = [torch.from_numpy(v.view(np.uint8).copy()).cuda() for v in verts]
    torch.cuda.synchronize()

    def loop(pipeline):
        ctx = rtdx.Context(W, H, bounces=bounces)
        up = ctx.upload_scene(sc)
        ctx.set_option(rtdx.OPT_PASS_PIPELINE, pipeline); ctx.set_option(rtdx.OPT_FRAME_PIPELINE, pipeline)
        pinned = [torch.empty((H, W, 4), dtype=torch.uint8).pin_memory().numpy() for _ in range(2)]
        images = []
        for f in range(n_frames):
            ctx.update_model_device(m, dev[f], base.size)
            ctx.collect_emissive_triangles()
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
        _, osc, _ = oracle_update(orc, sc, up["props"], m, verts[f], rtdx=rtdx)
        osc.render_threads(up["camera"], W, H, f, 1, 16, bounces=bounces, flags=0, accum=ref)
        osc.close()
    assert (bits(acc_on) != bits(ref)).sum() == 0


def test_steady_state_collect_neither_waits_nor_allocates(rtdx):
    """A collect after a device refit, queued behind a long sleep on the context stream, returns on the host while the sleep still
    runs; free device memory is the same before and after a series of such calls."""
    import torch
    sc = rtdx.scenes.instanced_blobs(n_models=2, lattice=4, emissive_fraction=0.25)
    m = len(sc.models) - 1
    stream = torch.cuda.Stream()
    ctx = rtdx.Context(32, 32, stream=stream.cuda_stream)
    ctx.upload_scene(sc)
    base = sc.models[m]["vertices"]
    dev = [_tensor(rtdx.scenes.deform(base, 0.1 * k, 0.3, seed=4)) for k in range(3)]
    ctx.collect_emissive_triangles()                 # the index and the buffers
    ctx.update_model_device(m, dev[0], base.size); ctx.collect_emissive_triangles()
    ctx.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for k in range(6):
        ctx.update_model_device(m, dev[k % 3], base.size); ctx.collect_emissive_triangles()
    ctx.synchronize()
    assert torch.cuda.mem_get_info()[0] == free0
    with torch.cuda.stream(stream):
        torch.cuda._sleep(4_000_000_000)             # about two seconds at the B200's clock
    t0 = time.perf_counter()
    n = ctx.collect_emissive_triangles()
    host_s = time.perf_counter() - t0
    busy = not stream.query()
    stream.synchronize()
    slept_s = time.perf_counter() - t0
    assert busy and host_s < 0.1 * slept_s, (host_s, slept_s)
    _collect_and_check(rtdx, ctx, with_vertices(sc, m, rtdx.scenes.deform(base, 0.2, 0.3, seed=4)), "after the sleep")
    assert n == ctx.read_emissive_triangles().size
    ctx.close()
