"""-m gpu parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.
Bar (BASELINE.json north_star): hit instance/primitive IDs bit-exact; here t,u,v and the accumulated radiance are
bit-exact as well (tolerance 0) because both sides fix the fp32 operation order (oracle/det_math.h, csrc/dmath.cuh)."""
import numpy as np
import pytest

from util import bits, compare_hits, hostile_material_scene, host_inputs, random_rays

pytestmark = pytest.mark.gpu


def _upload(rtdx, scene, W, H, **kw):
    ctx = rtdx.Context(W, H, **kw)
    up = ctx.upload_scene(scene)
    return ctx, up


def _oracle(orc, scene, up):
    return orc.OracleScene(scene, up["props"], up["lights"])


def _assert_hits_equal(gpu, ref):
    r = compare_hits(gpu, ref)
    assert r["inst"] == 0 and r["prim"] == 0 and r["t"] == 0 and r["u"] == 0 and r["v"] == 0, r


def test_trace_cornell_camera_and_random(rtdx, orc):
    sc = rtdx.scenes.cornell()
    ctx, up = _upload(rtdx, sc, 256, 256)
    osc = _oracle(orc, sc, up)
    rays = rtdx.scenes.camera_rays(up["camera"], 256, 256)
    _assert_hits_equal(ctx.trace(rays), osc.trace(rays, mode=0))
    rng = np.random.RandomState(7)
    rays = random_rays(rtdx, rng, 200000, (-1, 0, -1), (1, 2, 1))
    ref = osc.trace(rays, mode=0)
    _assert_hits_equal(ctx.trace(rays), ref)
    # any-hit agrees with "closest exists"
    ah = ctx.trace(rays, any_hit=True)
    assert np.array_equal(ah["inst"] != rtdx.MISS, ref["inst"] != rtdx.MISS)
    ctx.close()


def test_trace_edge_cases(rtdx, orc):
    sc = rtdx.scenes.cornell()
    ctx, up = _upload(rtdx, sc, 64, 64)
    osc = _oracle(orc, sc, up)
    assert ctx.trace(np.zeros(0, dtype=rtdx.ray_dt)).size == 0            # empty batch
    rays = np.zeros(6, dtype=rtdx.ray_dt)
    rays["origin"] = (0, 1, 0)
    rays["direction"] = [(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]   # axis-aligned, d has zeros
    rays["tmin"] = 1e-4
    rays["tmax"] = 1e4
    _assert_hits_equal(ctx.trace(rays), osc.trace(rays, mode=0))
    rays["tmax"] = 0.01                                                     # TMax before any surface
    assert (ctx.trace(rays)["inst"] == rtdx.MISS).all()
    rays["tmax"] = 0.5                                                      # TMax cuts some of the hits
    _assert_hits_equal(ctx.trace(rays), osc.trace(rays, mode=0))
    # negative zeros in the direction: the slab test must treat -0 like a (tiny) negative component, never cull a hit
    rays["origin"] = (0.1, 1.0, 0.05)
    rays["tmin"] = 1e-4
    rays["tmax"] = 1e4
    rays["direction"] = [(1, -0.0, -0.0), (-1, -0.0, 0.0), (-0.0, 1, -0.0), (-0.0, -1, -0.0), (-0.0, -0.0, 1), (0.0, -0.0, -1)]
    ref = osc.trace(rays, mode=0)
    assert (ref["inst"] != rtdx.MISS).sum() == 5                            # +z leaves through the open front of the box
    _assert_hits_equal(ctx.trace(rays), ref)
    assert np.array_equal(ctx.trace(rays, any_hit=True)["inst"] != rtdx.MISS, ref["inst"] != rtdx.MISS)
    # rays starting exactly on a surface with TMin = s_bias (the reference's bounce convention)
    rays["origin"] = (0.3, 0.0, 0.2)
    rays["tmin"] = 2e-5
    rays["tmax"] = 1e4
    _assert_hits_equal(ctx.trace(rays), osc.trace(rays, mode=0))
    ctx.close()


def test_trace_fuzz_degenerate_geometry_and_rays(rtdx, orc):
    """Hostile inputs against the brute-force definition (oracle mode 0): duplicated and zero-area triangles, coincident instances
    (equal t: the tie goes to the lowest instance, then primitive id), mirrored / non-uniformly scaled / sheared instance
    transforms, and rays with zero, denormal, huge, infinite and NaN components, TMin >= TMax, zero-length directions."""
    rng = np.random.RandomState(5)
    sc = rtdx.scenes.SceneDesc(); sc.name = "fuzz"
    sc.materials = np.concatenate([rtdx.scenes.default_material(), rtdx.scenes.make_material((.5, .5, .5))])
    nv = 60
    pos = rng.uniform(-1, 1, size=(nv, 3)).astype(np.float32)
    pos[:10] = np.round(pos[:10] * 4) / 4                                   # lattice points: exact edge / vertex hits happen
    tri = rng.randint(0, nv, size=(80, 3))
    tri[5] = tri[4]                                                         # duplicate triangle (tie on t)
    tri[6] = (tri[6][0], tri[6][0], tri[6][1])                              # zero-area triangles
    tri[7] = (3, 3, 3)
    m0 = sc.add_model(pos, np.zeros_like(pos), tri, np.full(80, 1))
    quad = np.array([[-2, -2, 0], [2, -2, 0], [2, 2, 0], [-2, 2, 0]], dtype=np.float32)
    m1 = sc.add_model(quad, np.zeros_like(quad), np.array([[0, 1, 2], [0, 2, 3]]), np.full(2, 1))
    eye = np.eye(4)
    mirror = np.diag([-1.0, 1.0, 1.0, 1.0])
    squash = np.diag([3.0, 0.25, 1.5, 1.0]); squash[:3, 3] = (0.5, -0.25, 0.125)
    shear = np.eye(4); shear[0, 1] = 0.75; shear[2, 0] = -0.5; shear[:3, 3] = (-1, 0.5, 2)
    for m in (eye, eye, mirror, squash, shear):                             # instances 0 and 1 coincide exactly
        sc.add_instance(m0, m)
    back = np.eye(4); back[2, 3] = -1.5
    sc.add_instance(m1, back); sc.add_instance(m1, back)                    # two coincident quads
    ctx, up = _upload(rtdx, sc, 16, 16)
    osc = _oracle(orc, sc, up)
    n = 20000
    rays = random_rays(rtdx, rng, n, (-3, -3, -3), (3, 3, 3))
    rays["origin"][:2000] = pos[rng.randint(0, nv, 2000)] + np.float32(2.0) * rays["direction"][:2000] * -1     # aimed at vertices
    d = rays["direction"]
    d[2000:2400, 0] = 0.0; d[2400:2800, 1] = -0.0; d[2800:3000, :2] = 0.0                                          # axis-parallel, +-0
    d[3000:3100] *= np.float32(1e-30); d[3100:3200] *= np.float32(1e30); d[3200:3300] *= np.float32(1e-42)        # tiny / huge / denormal lengths
    d[3300:3320] = 0.0                                                                                             # zero direction
    d[3320:3340, 0] = np.nan; d[3340:3360, 1] = np.inf; rays["origin"][3360:3380, 2] = np.nan; rays["origin"][3380:3400, 0] = -np.inf
    rays["tmin"][3400:3500] = 1.0; rays["tmax"][3400:3500] = 1.0                                                   # empty interval
    rays["tmin"][3500:3600] = 2.0; rays["tmax"][3500:3600] = 1.0                                                   # inverted interval
    rays["tmin"][3600:3700] = 0.0; rays["tmax"][3600:3700] = np.inf
    rays["origin"][3700:3800] *= np.float32(1e6)                                                                   # far away
    ref = osc.trace(rays, mode=0)
    g = ctx.trace(rays)
    _assert_hits_equal(g, ref)
    assert (ref["inst"] != rtdx.MISS).sum() > 3000
    ah = ctx.trace(rays, any_hit=True)
    assert np.array_equal(ah["inst"] != rtdx.MISS, ref["inst"] != rtdx.MISS)
    ctx.close()


@pytest.mark.parametrize("n_side", [8, 40])
def test_trace_mesh_room(rtdx, orc, n_side):
    sc = rtdx.scenes.mesh_room(n=n_side)
    ctx, up = _upload(rtdx, sc, 128, 128)
    osc = _oracle(orc, sc, up)
    rng = np.random.RandomState(11)
    rays = np.concatenate([rtdx.scenes.camera_rays(up["camera"], 128, 128), random_rays(rtdx, rng, 100000, (-5, 0.1, -5), (5, 5.9, 5))])
    ref = osc.trace(rays, mode=1)
    _assert_hits_equal(ctx.trace(rays), ref)
    sub = rays[:4000]
    _assert_hits_equal(osc.trace(sub, mode=1), osc.trace(sub, mode=0))     # oracle BVH2 == brute force
    ctx.close()


def test_trace_instanced(rtdx, orc):
    sc = rtdx.scenes.instanced_blobs(n_models=3, n_side=6, lattice=4)
    ctx, up = _upload(rtdx, sc, 128, 128)
    osc = _oracle(orc, sc, up)
    rng = np.random.RandomState(13)
    rays = np.concatenate([rtdx.scenes.camera_rays(up["camera"], 128, 128), random_rays(rtdx, rng, 50000, (-2.5, -2.5, -2.5), (2.5, 2.5, 2.5))])
    ref = osc.trace(rays, mode=1)
    _assert_hits_equal(ctx.trace(rays), ref)
    sub = rays[::37]
    _assert_hits_equal(osc.trace(sub, mode=1), osc.trace(sub, mode=0))
    ctx.close()


def _render_both(rtdx, orc, sc, W, H, spp, bounces, flags, spp_per_pass=1, step=1):
    ctx, up = _upload(rtdx, sc, W, H, bounces=bounces, flags=flags, samples_per_pass=spp_per_pass)
    osc = _oracle(orc, sc, up)
    ctx.reset_counters()
    ctx.render_pass(0, spp)
    ctx.synchronize()
    gpu = ctx.read_accum()
    cnt = ctx.counters()
    ref, octr = osc.render(up["camera"], W, H, 0, spp, bounces=bounces, flags=flags, step=step)
    return ctx, gpu, cnt, ref, octr


def test_render_cornell_c1_bit_exact(rtdx, orc):
    """BASELINE config C1: Cornell 36 tris, 256x256, 16 spp, depth 4 (bounces=2), Lambert only, jitter on."""
    sc = rtdx.scenes.cornell()
    flags = rtdx.FLAG_JITTER | rtdx.FLAG_LAMBERT_ONLY
    ctx, gpu, cnt, ref, octr = _render_both(rtdx, orc, sc, 256, 256, 16, 2, flags, spp_per_pass=4)
    assert cnt["closest_rays"] == octr["closest_rays"] and cnt["shadow_rays"] == octr["shadow_rays"], (cnt, octr)
    mism = bits(gpu) != bits(ref)
    assert mism.sum() == 0, "radiance mismatches: %d of %d floats" % (mism.sum(), mism.size)
    # output image (F20)
    assert np.array_equal(ctx.read_output(), orc.resolve(ref))
    ctx.close()


def test_render_mesh_room_ggx(rtdx, orc):
    """C2-shaped (GGX + diffuse, smooth normals, two instances) at a size the oracle finishes in seconds."""
    sc = rtdx.scenes.mesh_room(n=24)
    ctx, gpu, cnt, ref, octr = _render_both(rtdx, orc, sc, 96, 64, 2, 6, 0)
    assert cnt["closest_rays"] == octr["closest_rays"] and cnt["shadow_rays"] == octr["shadow_rays"], (cnt, octr)
    mism = bits(gpu) != bits(ref)
    assert mism.sum() == 0, "radiance mismatches: %d of %d floats" % (mism.sum(), mism.size)
    ctx.close()


def test_render_instanced_emitters(rtdx, orc):
    """C3-shaped: TLAS over rotated/scaled instances, many emissive triangles, NEE."""
    sc = rtdx.scenes.instanced_blobs(n_models=3, n_side=6, lattice=4, emissive_fraction=0.1)
    ctx, gpu, cnt, ref, octr = _render_both(rtdx, orc, sc, 96, 64, 2, 3, 0)
    assert cnt["closest_rays"] == octr["closest_rays"] and cnt["shadow_rays"] == octr["shadow_rays"], (cnt, octr)
    mism = bits(gpu) != bits(ref)
    assert mism.sum() == 0, "radiance mismatches: %d of %d floats" % (mism.sum(), mism.size)
    ctx.close()


def _restir_frames(rtdx, orc, sc, W, H, bounces, flags, script):
    """Runs the reference's 3-pass frame (RayGen, RayGen2, RayGen3) on the engine and on the oracle for a script of frames:
    each entry is (camera or None, instance transforms or None) applied before the frame.  Everything is compared bit-exactly."""
    ctx, up = _upload(rtdx, sc, W, H, bounces=bounces, flags=flags | rtdx.FLAG_RESTIR)
    osc = _oracle(orc, sc, up)
    frames = osc.new_frames(W, H)
    acc = np.zeros((H, W, 4), dtype=np.float32)
    cam = up["camera"]
    model_ids = [i[0] for i in sc.instances]
    total = {"closest_rays": 0, "shadow_rays": 0}
    ctx.reset_counters()
    for f, (new_cam, xforms) in enumerate(script):
        if xforms is not None:                                      # OnUpdate: UpdateInstancePropertiesBuffer + TLAS refit
            props, descs = rtdx.instance_properties(xforms, [up["model_ids"][m] for m in model_ids])
            if f > 0:
                props["prevObjectToWorld"] = prev_props["objectToWorld"]; props["prevObjectToWorldInverse"] = prev_props["objectToWorldInverse"]
                props["prevObjectToWorldNormal"] = prev_props["objectToWorldNormal"]
            ctx.set_instances(descs, props)
            ctx.set_emissive_triangles(up["lights"])
            osc.set_props(props)
            prev_props = props
        elif f == 0:
            prev_props = up["props"]
        if new_cam is not None:                                     # UpdateCameraBuffer: prevView / prevProjection = last frame's
            new_cam = new_cam.copy()
            new_cam["prevView"] = cam["view"]; new_cam["prevProjection"] = cam["projection"]
            if np.abs(new_cam["view"] - cam["view"]).max() > 2e-5:
                acc[:] = 0                                           # Pass_spat_di_v7.hlsl:407-423
            cam = new_cam
            ctx.set_camera(cam)
        ctx.render_frame(f)
        ctx.synchronize()
        octr = osc.render_frame(cam, W, H, f, frames, acc, bounces=bounces, flags=flags)
        for k in total:
            total[k] += octr[k]
        gpu, cnt = ctx.read_accum(), ctx.counters()
        assert (cnt["closest_rays"], cnt["shadow_rays"]) == (total["closest_rays"], total["shadow_rays"]), (f, cnt, total)
        rs_g, rs_o = ctx.read_restir(), osc.dump_frames(frames, W, H)
        bad = (bits(rs_g) != bits(rs_o)).any(axis=-1)
        assert bad.sum() == 0, "frame %d: %d pixels with differing reservoirs, first %s" % (f, bad.sum(), np.argwhere(bad)[:3])
        mism = bits(gpu) != bits(acc)
        assert mism.sum() == 0, "frame %d: %d accumulation floats differ" % (f, mism.sum())
    stats = {"M_di_mean": float(rs_o[..., 11].mean()), "M_gi_mean": float(rs_o[..., 23].mean())}
    osc.free_frames(frames)
    ctx.close()
    return stats


def test_restir_static_frames_bit_exact(rtdx, orc):
    """SURVEY §8f rank 1: temporal + spatial reuse.  Static camera and scene: reprojection lands on the same pixel, M grows
    to the temporal cap, reservoirs / ray counts / accumulation equal the oracle's on every frame."""
    sc = rtdx.scenes.cornell()
    st = _restir_frames(rtdx, orc, sc, 96, 80, 2, 0, [(None, None)] * 4)
    assert st["M_di_mean"] > 8.0                                    # history was actually reused
    sc = rtdx.scenes.mesh_room(n=16)
    _restir_frames(rtdx, orc, sc, 80, 48, 3, 0, [(None, None)] * 3)


def test_restir_moving_camera_and_instances_bit_exact(rtdx, orc):
    """Camera motion (reprojection through prevView/prevProjection, accumulation reset) and instance motion
    (reprojection through objectToWorldInverse / prevObjectToWorld, TLAS refit per frame, Renderer.cpp:444-449,594)."""
    sc = rtdx.scenes.cornell()
    cams = [None, rtdx.camera_params((sc.eye[0] + 0.05, sc.eye[1], sc.eye[2]), sc.center, sc.up, 96 / 80.0),
            rtdx.camera_params((sc.eye[0] + 0.10, sc.eye[1] + 0.02, sc.eye[2]), sc.center, sc.up, 96 / 80.0), None]
    _restir_frames(rtdx, orc, sc, 96, 80, 2, 0, [(c, None) for c in cams])
    sc = rtdx.scenes.instanced_blobs(n_models=2, n_side=5, lattice=3, emissive_fraction=0.15)
    base = [np.asarray(i[1], dtype=np.float64).reshape(4, 4).T for i in sc.instances]     # column-vector 4x4

    def moved(t):
        out = []
        for k, m in enumerate(base):
            m2 = m.copy()
            if k % 2 == 0:
                m2[0, 3] += 0.05 * t
            out.append(m2)
        return [rtdx.xmmatrix_from_colvec(m) for m in out]
    _restir_frames(rtdx, orc, sc, 80, 64, 3, 0, [(None, moved(t)) for t in range(3)])


def test_restir_frames_in_concurrent_parts(rtdx, orc):
    """The ReSTIR frame's first pass runs as concurrent path ranges too (>= 65536 paths): reservoirs, ray counts and the accumulation of
    three frames are bit-identical for 1, 2 and 3 parts, and frame 0 (no history: E0 of the fresh reservoirs) equals the oracle."""
    sc = rtdx.scenes.mesh_room(n=16)
    W, H, bounces = 384, 192, 2                                      # 73 728 paths
    ref = None
    for parts in (1, 2, 3):
        ctx, up = _upload(rtdx, sc, W, H, bounces=bounces, flags=rtdx.FLAG_RESTIR)
        ctx.set_option(rtdx.OPT_PASS_PARTS, parts)
        ctx.reset_counters()
        out = []
        for f in range(3):
            ctx.render_frame(f); ctx.synchronize()
            out.append((ctx.read_restir(), ctx.read_accum(), ctx.counters()))
        if ref is None:
            ref = out
            osc = _oracle(orc, sc, up)
            frames = osc.new_frames(W, H)
            acc = np.zeros((H, W, 4), dtype=np.float32)
            octr = osc.render_frame(up["camera"], W, H, 0, frames, acc, bounces=bounces, flags=0)
            assert (out[0][2]["closest_rays"], out[0][2]["shadow_rays"]) == (octr["closest_rays"], octr["shadow_rays"])
            assert np.array_equal(bits(out[0][0]), bits(osc.dump_frames(frames, W, H))) and np.array_equal(bits(out[0][1]), bits(acc))
            osc.free_frames(frames)
        else:
            for f in range(3):
                assert np.array_equal(bits(out[f][0]), bits(ref[f][0])), (parts, f)
                assert np.array_equal(bits(out[f][1]), bits(ref[f][1])), (parts, f)
                assert (out[f][2]["closest_rays"], out[f][2]["shadow_rays"]) == (ref[f][2]["closest_rays"], ref[f][2]["shadow_rays"]), (parts, f)
        ctx.close()


@pytest.mark.parametrize("scene_name", ["cornell", "mesh", "inst"])
def test_legacy_rr_estimator_bit_exact(rtdx, orc, scene_name):
    """RTX_FLAG_LEGACY_RR (SURVEY 8f rank 4): the reference's older estimator (include/RayGen.hlsl + include/Hit.hlsl: RIS-10 NEE with one
    shadow ray per bounce, MIS on emitter hits, Russian roulette after depth 3, fp32 materials, face-forwarded normals) as a wavefront;
    ray counts and accumulated radiance bit-identical to the oracle's restatement, 2 passes of 2 samples."""
    sc = {"cornell": lambda: rtdx.scenes.cornell(), "mesh": lambda: rtdx.scenes.mesh_room(n=20),
          "inst": lambda: rtdx.scenes.instanced_blobs(n_models=3, n_side=6, lattice=3, emissive_fraction=0.2)}[scene_name]()
    W, H, bounces = 96, 64, 12
    flags = rtdx.FLAG_LEGACY_RR
    ctx = rtdx.Context(W, H, bounces=bounces, flags=flags, samples_per_pass=2)
    up = ctx.upload_scene(sc)
    osc = orc.OracleScene(sc, up["props"], up["lights"])
    ctx.render_pass(0, 2); ctx.render_pass(2, 2); ctx.synchronize()
    cnt = ctx.counters()
    ref, octr = osc.render(up["camera"], W, H, 0, 4, bounces=bounces, flags=flags)
    assert cnt["closest_rays"] == octr["closest_rays"] and cnt["shadow_rays"] == octr["shadow_rays"] and cnt["paths"] == octr["paths"], (cnt, octr)
    gpu = ctx.read_accum()
    assert (bits(gpu) != bits(ref)).sum() == 0
    assert gpu[..., 3].mean() > 0.9 * 4 and np.isfinite(gpu).all() and gpu[..., :3].sum() > 0       # the estimator produces light
    if scene_name == "mesh":                                                                        # closed room: paths end by RR / emitter hits,
        assert 4.5 * W * H * 4 < octr["closest_rays"] < 0.9 * bounces * W * H * 4                   # not by the cap
    ctx.close()


def test_engine_side_reduce_single_rank(rtdx):
    """rtx_comm_init / rtx_reduce_accum / rtx_read_reduced_accum with a communicator of one rank (NCCL bound at run time): the reduced
    buffer equals the context's own accumulation after every pass, rtx_read_output resolves it, and rendering continues to accumulate
    (the next pass's accumulation waits for the reduce, not the other way round).  Two ranks: tests/test_gpu_host.py, bench.py --gpus N."""
    sc = rtdx.scenes.cornell()
    W, H = 64, 48
    ctx, up = _upload(rtdx, sc, W, H, bounces=2)
    ref, _ = _upload(rtdx, sc, W, H, bounces=2)
    ctx.comm_init(ctx.comm_unique_id(), 0, 1)
    for k in range(3):
        ctx.render_pass(k, 1); ctx.reduce_accum()
        ref.render_pass(k, 1); ref.synchronize()
        total = ctx.read_reduced_accum()
        assert np.array_equal(bits(total), bits(ref.read_accum())), k
        assert np.array_equal(ctx.read_output(), ref.read_output())
    ctx.close(); ref.close()


def test_builder_quality_and_shape(rtdx):
    """The GPU builder (Morton -> PLOC with the SAH programme -> 8-wide collapse) beyond "the hits are right": node fan-out, leaf size,
    SAH cost and the per-ray work it leads to stay inside bounds a regression in any stage would break; a TLAS holds ONE instance per leaf
    slot (a ray enters only the instances whose own boxes it hits)."""
    sc = rtdx.scenes.mesh_room(n=64)                      # 49 152 triangles + the 14-triangle room
    ctx, up = _upload(rtdx, sc, 256, 144)
    info = ctx.blas_info(up["model_ids"][0])
    n_tris = sc.models[0]["indices"].size // 3
    assert info["n_tris"] == n_tris
    assert n_tris / 24 <= info["n_nodes"] <= n_tris / 4          # 8 children of <= 3 triangles: between full and a quarter full
    assert 0.5 < info["build_ms"] < 2000
    rays = rtdx.scenes.camera_rays(up["camera"], 256, 144)
    import torch
    r = torch.from_numpy(rays.view(np.float32).reshape(-1, 8)).cuda(); h = torch.empty((r.shape[0], 5), dtype=torch.float32, device="cuda")
    ctx.reset_counters(); ctx.trace_device(r.data_ptr(), r.shape[0], h.data_ptr(), stats=True); ctx.synchronize()
    c = ctx.counters(); n = r.shape[0]
    nodes, tris, inst = c["nodes_visited"] / n, c["tris_tested"] / n, c["instances_entered"] / n
    assert nodes < 9.0 and tris < 8.0, (nodes, tris)             # measured 5.3 / 4.9: a broken SAH collapse or slot order doubles them
    assert 1.0 <= inst < 1.6                                     # the room always, the mesh only when its own box is hit (round 1: 2.000)
    ctx.close()
    sc = rtdx.scenes.instanced_blobs(n_models=3, n_side=6, lattice=6)      # 216 instances: a multi-level TLAS
    ctx, up = _upload(rtdx, sc, 128, 128)
    rays = rtdx.scenes.camera_rays(up["camera"], 128, 128)
    r = torch.from_numpy(rays.view(np.float32).reshape(-1, 8)).cuda(); h = torch.empty((r.shape[0], 5), dtype=torch.float32, device="cuda")
    ctx.reset_counters(); ctx.trace_device(r.data_ptr(), r.shape[0], h.data_ptr(), stats=True); ctx.synchronize()
    c = ctx.counters()
    hit = (h[:, 4].view(torch.int32) != -1).float().mean().item()
    assert c["instances_entered"] / r.shape[0] < 1.5 + 2.0 * hit  # a few instance records per ray that hits something, not the leaf's neighbours too
    ctx.close()


def test_call_order_violations_return_state_errors_not_faults(rtdx):
    """ADVICE r1 (medium): rtx_upload_model after rtx_set_instances invalidates the per-model tables; rendering or tracing before the
    next rtx_set_instances must fail with RTX_ERR_STATE, not hand freed tables to the kernels — and the context stays usable."""
    sc = rtdx.scenes.cornell()
    ctx, up = _upload(rtdx, sc, 32, 32, bounces=2)
    ctx.render_pass(0, 1); ctx.synchronize()
    m = sc.models[0]
    ctx.upload_model(m["vertices"], m["indices"], m["material_id_offset"])           # a second model arrives late
    for call in (lambda: ctx.render_pass(1, 1), lambda: ctx.trace(rtdx.scenes.camera_rays(up["camera"], 8, 8))):
        with pytest.raises(rtdx.RtxError) as e:
            call()
        assert "rtx error 3" in str(e.value)
    ctx.set_instances(up["descs"], up["props"])                                       # OnUpdate again: everything is valid again
    ctx.reset_accum(); ctx.render_pass(0, 1); ctx.synchronize()
    a = ctx.read_accum()
    ctx2, _ = _upload(rtdx, sc, 32, 32, bounces=2)
    ctx2.render_pass(0, 1); ctx2.synchronize()
    assert np.array_equal(bits(a), bits(ctx2.read_accum()))
    ctx.close(); ctx2.close()


def test_fast_math_mode_converges_to_the_exact_image(rtdx, orc):
    """RTX_FLAG_FAST_MATH (shading stages built with FMA contraction and approximate div / sqrt / rsqrt / sincos): not bit-identical —
    a path diverges where a rounding flips a discrete decision — but the same estimator: BASELINE.json asks for radiance "within a
    stated relative tolerance, with mean-image RMSE reported".  Stated here, at 256 spp against the exact mode (which is bit-identical
    to the oracle, checked on the first samples): mean-image difference < 0.2 %, RMSE of the per-pixel means < 1 % of the image mean
    (measured: 0.0002 % and 0.15 %), fewer than 0.5 % of the pixels further than 20 % apart; ray counts within 0.1 %."""
    sc = rtdx.scenes.mesh_room(n=24)
    W, H, SPP, B = 96, 64, 256, 6
    imgs, cnts = {}, {}
    for name, flags in (("exact", 0), ("fast", rtdx.FLAG_FAST_MATH)):
        ctx, up = _upload(rtdx, sc, W, H, bounces=B, flags=flags, samples_per_pass=8)
        ctx.reset_counters()
        ctx.render_pass(0, 2); ctx.synchronize()
        first = ctx.read_accum()
        if name == "exact":
            ref, _ = _oracle(orc, sc, up).render(up["camera"], W, H, 0, 2, bounces=B)
            assert (bits(first) != bits(ref)).sum() == 0
        else:
            assert (bits(first) != bits(imgs["exact_first"])).sum() > 0          # it IS a different arithmetic
        imgs[name + "_first"] = first
        ctx.render_pass(2, SPP - 2); ctx.synchronize()
        a = ctx.read_accum()
        assert (a[..., 3] == SPP).all()
        imgs[name] = a[..., :3] / a[..., 3:4]
        cnts[name] = ctx.counters()
        ctx.close()
    e, f = imgs["exact"].astype(np.float64), imgs["fast"].astype(np.float64)
    mean = e.mean()
    rel_mean = abs(f.mean() - mean) / mean
    rmse = np.sqrt(((e - f) ** 2).mean()) / mean
    lum_e, lum_f = e.mean(-1), f.mean(-1)
    far = (np.abs(lum_e - lum_f) > 0.2 * np.maximum(lum_e, 1e-3)).mean()
    print("fast math vs exact at %d spp: mean-image difference %.4f %%, RMSE %.3f %% of the mean, %.2f %% of the pixels > 20 %% apart" % (
        SPP, 100 * rel_mean, 100 * rmse, 100 * far))
    assert rel_mean < 0.002 and rmse < 0.01 and far < 0.005, (rel_mean, rmse, far)
    for k in ("closest_rays", "shadow_rays"):
        assert abs(cnts["fast"][k] - cnts["exact"][k]) < 1e-3 * cnts["exact"][k]


def test_async_readback_and_frame_in_flight_match_blocking_calls(rtdx):
    """rtx_read_output_async / rtx_wait_output with one frame in flight (bench.py's e2e loop) give the images of the blocking per-frame
    loop: same RGBA8 bytes after every frame, with rtx_set_instances / rtx_set_camera called every frame in both loops."""
    sc = rtdx.scenes.mesh_room(n=12)
    W, H = 128, 96
    imgs = []
    for mode in ("blocking", "in_flight"):
        ctx, up = _upload(rtdx, sc, W, H, bounces=2)
        outs = [np.zeros((H, W, 4), dtype=np.uint8) for _ in range(2)]
        got = []
        for k in range(4):
            ctx.set_instances(up["descs"], up["props"])
            ctx.set_camera(up["camera"])
            ctx.render_pass(k, 1)
            if mode == "blocking":
                got.append(ctx.read_output().copy())
            else:
                ctx.wait_output()
                if k > 0:
                    got.append(outs[(k - 1) & 1].copy())
                ctx.read_output_async(outs[k & 1])
        if mode == "in_flight":
            ctx.wait_output(); got.append(outs[3 & 1].copy())
        imgs.append(got)
        ctx.close()
    for a, b in zip(*imgs):
        assert np.array_equal(a, b)
    assert imgs[0][3].any() and not np.array_equal(imgs[0][0], imgs[0][3])


def test_instance_list_changes_between_frames(rtdx, orc):
    """rtx_set_instances through its three paths — rebuild (count or models changed), refit (same models), one-node rewrite (<= 3
    instances) — in one context: the instance list shrinks, is permuted to other models, and grows back; hits equal the oracle each time."""
    sc = rtdx.scenes.instanced_blobs(n_models=3, n_side=5, lattice=3, emissive_fraction=0.1)      # 27 instances
    W, H = 48, 32
    ctx, up = _upload(rtdx, sc, W, H)
    osc = _oracle(orc, sc, up)
    rng = np.random.RandomState(9)
    rays = np.concatenate([rtdx.scenes.camera_rays(up["camera"], W, H), random_rays(rtdx, rng, 8000, -5.0, 5.0)])
    all_models = [i[0] for i in sc.instances]
    all_xf = [np.asarray(i[1], dtype=np.float32) for i in sc.instances]
    n_models = max(all_models) + 1
    for pick, shift in ((range(27), 0), (range(0, 27, 4), 0), (range(0, 27, 4), 1), (range(2), 0), (range(3), 1), (range(27), 1), (range(27), 1)):
        idx = list(pick)
        models = [(all_models[i] + shift) % n_models for i in idx]
        props, descs = rtdx.instance_properties([all_xf[i] for i in idx], [up["model_ids"][m] for m in models])
        ctx.set_instances(descs, props)
        got = ctx.trace(rays)
        osc._model_ids = models
        osc.set_props(props)
        _assert_hits_equal(got, osc.trace(rays, mode=1))
    ctx.close()


def test_resolve_source_external_accumulation_buffer(rtdx):
    """rtx_set_resolve_source: rank 0 of a multi-GPU job resolves the reduced accumulation buffer instead of its private partial sum."""
    import importlib
    import torch
    wrap = importlib.import_module("royaltracer-dx_b200.dist").wrap_device_buffer
    sc = rtdx.scenes.cornell()
    W, H = 96, 64
    ctx, up = _upload(rtdx, sc, W, H, bounces=2)
    ctx.render_pass(0, 1); img0 = ctx.read_output().copy()
    saved = wrap(ctx.accum_device_ptr(), (H, W, 4)).clone()
    ctx.render_pass(1, 1); img1 = ctx.read_output().copy()
    assert not np.array_equal(img0, img1)
    ctx.set_resolve_source(saved.data_ptr())
    assert np.array_equal(ctx.read_output(), img0)
    ctx.set_resolve_source(None)
    assert np.array_equal(ctx.read_output(), img1)
    torch.cuda.synchronize()
    ctx.close()


def test_tlas_refit_matches_rebuild_and_oracle(rtdx, orc):
    """Per-frame TLAS refit (rdn/Renderer.cpp:594): rtx_set_instances keeps the topology of the last build and refits the node boxes on
    the stream; hits after large seeded instance motion equal those of a forced rebuild (RTX_OPT_TLAS_REBUILD) and of the oracle."""
    sc = rtdx.scenes.instanced_blobs(n_models=3, n_side=6, lattice=4, emissive_fraction=0.1)      # 64 instances
    W, H = 64, 48
    ctx, up = _upload(rtdx, sc, W, H)
    osc = _oracle(orc, sc, up)
    model_ids = [i[0] for i in sc.instances]
    base = [np.asarray(i[1], dtype=np.float64).reshape(4, 4).T for i in sc.instances]
    rng = np.random.RandomState(5)
    rays = np.concatenate([rtdx.scenes.camera_rays(up["camera"], W, H), random_rays(rtdx, rng, 20000, -6.0, 6.0)])
    for t in range(1, 4):
        xf = []
        for k, m in enumerate(base):
            a = 0.7 * t * rng.uniform(-1, 1)
            R = np.array([[np.cos(a), 0, np.sin(a), 0], [0, 1, 0, 0], [-np.sin(a), 0, np.cos(a), 0], [0, 0, 0, 1]])
            m2 = m @ R
            m2[:3, 3] += rng.uniform(-0.8, 0.8, 3) * t
            xf.append(rtdx.xmmatrix_from_colvec(m2))
        props, descs = rtdx.instance_properties(xf, [up["model_ids"][m] for m in model_ids])
        ctx.set_option(rtdx.OPT_TLAS_REBUILD, 0)
        ctx.set_instances(descs, props)
        h_refit = ctx.trace(rays)
        ctx.set_option(rtdx.OPT_TLAS_REBUILD, 1)
        ctx.set_instances(descs, props)
        h_build = ctx.trace(rays)
        for k in ("inst", "prim", "t", "u", "v"):
            assert np.array_equal(h_refit[k].view(np.uint32), h_build[k].view(np.uint32)), (t, k)
        osc.set_props(props)
        _assert_hits_equal(h_refit, osc.trace(rays, mode=1))
        assert (h_refit["inst"] != rtdx.MISS).mean() > 0.05
    ctx.close()


def test_interleaved_and_contiguous_pass_parts_match_the_oracle(rtdx, orc):
    """RTX_OPT_PASS_PARTS: a pass of >= 65536 paths is cut into path ranges (interleaved chunks of image rows when a chunk of <= 32 rows
    divides the frame evenly among the parts, else contiguous ranges) that run on separate CUDA streams; ray counts and the accumulated
    radiance stay bit-identical to the oracle for 1..4 parts (paths never interact before the accumulation)."""
    sc = rtdx.scenes.mesh_room(n=16)
    bounces = 3
    # 384 x 192 = 73 728 paths: every part count interleaves; 384 x 191 = 73 344 paths: 191 is prime, so the parts are contiguous ranges
    for (W, H), part_counts in (((384, 192), (1, 2, 3, 4)), ((384, 191), (2, 3, 4))):
        ctx, up = _upload(rtdx, sc, W, H, bounces=bounces)
        osc = orc.OracleScene(sc, up["props"], up["lights"])
        ref, octr = osc.render(up["camera"], W, H, 0, 1, bounces=bounces, flags=0)
        for parts in part_counts:
            ctx.set_option(rtdx.OPT_PASS_PARTS, parts)
            ctx.reset_accum(); ctx.reset_counters()
            ctx.render_pass(0, 1); ctx.synchronize()
            cnt = ctx.counters()
            assert cnt["closest_rays"] == octr["closest_rays"] and cnt["shadow_rays"] == octr["shadow_rays"], (W, H, parts, cnt, octr)
            assert (bits(ctx.read_accum()) != bits(ref)).sum() == 0, (W, H, parts)
        ctx.close()
    # several samples per pass: the paths of a pass are (sample, pixel) pairs, the chunks are cut in that space
    W2, H2, spp = 192, 96, 4                                                               # 73 728 paths again
    ctx, up = _upload(rtdx, sc, W2, H2, bounces=bounces, samples_per_pass=spp)
    ref2, octr2 = osc.render(up["camera"], W2, H2, 0, spp, bounces=bounces, flags=0)
    for parts in (1, 2, 3, 4):
        ctx.set_option(rtdx.OPT_PASS_PARTS, parts)
        ctx.reset_accum(); ctx.reset_counters()
        ctx.render_pass(0, spp); ctx.synchronize()
        cnt = ctx.counters()
        assert cnt["closest_rays"] == octr2["closest_rays"] and cnt["shadow_rays"] == octr2["shadow_rays"], (parts, cnt, octr2)
        assert (bits(ctx.read_accum()) != bits(ref2)).sum() == 0, parts
    ctx.close()


def test_graph_replay_shadow_stream_and_trace_order_do_not_change_the_image(rtdx, orc):
    """RTX_OPT_PASS_GRAPH: the third and later passes of a static configuration replay a captured CUDA graph (the sample index comes
    from a device word).  The DI visibility rays of a pass are traced on a side stream, or in sequence when RTX_OPT_TRACE_STATS is on
    (which also runs without a graph, as one part).  The traversal kernels claim rays longest-first through the queue's order array
    where the scene's heavy instances separate anything (mesh_room), and in emission order where they do not (cornell: one model, so
    its heavy box is the scene box).  For each scene six accumulated samples are bit-identical by default, with the graph off and with
    statistics on — and equal to the oracle's six samples; the kernel-launch count is the same whether a pass was launched directly or
    replayed."""
    W, H, bounces, n_samples = 384, 192, 3, 6
    for sc in (rtdx.scenes.mesh_room(n=16), rtdx.scenes.cornell()):
        ctx, up = _upload(rtdx, sc, W, H, bounces=bounces)
        osc = orc.OracleScene(sc, up["props"], up["lights"])
        ref = None
        for s in range(n_samples):
            img, _ = osc.render(up["camera"], W, H, s, 1, bounces=bounces, flags=0)
            ref = img if ref is None else ref + img               # gPermanentData += sample, in sample order (F20)
        results = {}
        # (name, options, path ranges per pass): a pass with statistics runs as one range
        for name, opts, parts in (("default", {}, 2), ("no graph", {rtdx.OPT_PASS_GRAPH: 0}, 2),
                                  ("statistics, shadow rays in sequence", {rtdx.OPT_TRACE_STATS: 1}, 1)):
            ctx.set_option(rtdx.OPT_PASS_GRAPH, 1); ctx.set_option(rtdx.OPT_TRACE_STATS, 0)
            for k, v in opts.items():
                ctx.set_option(k, v)
            ctx.reset_accum(); ctx.reset_counters()
            per_pass = []
            for s in range(n_samples):
                before = ctx.counters()["kernel_launches"]
                ctx.render_pass(s, 1)
                per_pass.append(ctx.counters()["kernel_launches"] - before)
            ctx.synchronize()
            results[name] = (ctx.read_accum(), ctx.counters(), per_pass)
            assert len(set(per_pass)) == 1 and per_pass[0] > 10 * parts, (sc.name, name, per_pass)
        base = results["default"]
        assert (bits(base[0]) != bits(ref)).sum() == 0, sc.name
        for name, (img, cnt, per_pass) in results.items():
            assert np.array_equal(bits(img), bits(base[0])), (sc.name, name)
            assert cnt["closest_rays"] == base[1]["closest_rays"] and cnt["shadow_rays"] == base[1]["shadow_rays"], (sc.name, name)
        ctx.close()


def test_set_option_rejects_unknown_options_and_part_counts(rtdx):
    """rtx_set_option fails with RTX_ERR_ARG for an option value no RTX_OPT_* names (among them 5..9, 11 and 12, which named launch
    tuning options once) and for a RTX_OPT_PASS_PARTS count outside 1..4; the context stays usable."""
    ctx, _ = _upload(rtdx, rtdx.scenes.cornell(), 64, 64, bounces=2)
    for option in (5, 6, 7, 8, 9, 11, 12, 0, 15):
        with pytest.raises(rtdx.RtxError, match="unknown option"):
            ctx.set_option(option, 1)
    for parts in (0, 5):
        with pytest.raises(rtdx.RtxError, match="RTX_OPT_PASS_PARTS"):
            ctx.set_option(rtdx.OPT_PASS_PARTS, parts)
    ctx.set_option(rtdx.OPT_PASS_PARTS, 4)
    ctx.render_pass(0, 1); ctx.synchronize()
    ctx.close()


def test_pipelined_passes_are_bit_identical(rtdx, orc):
    """RTX_OPT_PASS_PIPELINE: rtx_render_pass calls that directly follow each other alternate between two sets of pass buffers on two
    streams and overlap; gPermanentData is shared and the accumulations are chained in call order, so seven samples equal the oracle's
    seven samples bit for bit — back to back, through the n_samples loop of one call, with the pipeline off, with other calls
    (camera, engine-side reduce) between the passes — and a camera change in the middle of a sequence resets the accumulation at the
    right place."""
    sc = rtdx.scenes.mesh_room(n=16)
    W, H, bounces, n_samples = 384, 192, 3, 7
    ctx, up = _upload(rtdx, sc, W, H, bounces=bounces)
    osc = orc.OracleScene(sc, up["props"], up["lights"])
    ref, rays = None, [0, 0]
    per_sample = []
    for s in range(n_samples):
        img, octr = osc.render(up["camera"], W, H, s, 1, bounces=bounces, flags=0)
        per_sample.append(img)
        ref = img if ref is None else ref + img
        rays[0] += octr["closest_rays"]; rays[1] += octr["shadow_rays"]

    def check(tag):
        ctx.synchronize()
        cnt = ctx.counters()
        assert np.array_equal(bits(ctx.read_accum()), bits(ref)), tag
        assert (cnt["closest_rays"], cnt["shadow_rays"]) == tuple(rays), (tag, cnt, rays)

    for tag, pipeline in (("back to back", 1), ("pipeline off", 0)):
        ctx.set_option(rtdx.OPT_PASS_PIPELINE, pipeline)
        ctx.reset_accum(); ctx.reset_counters()
        for s in range(n_samples):
            ctx.render_pass(s, 1)
        check(tag)
    ctx.set_option(rtdx.OPT_PASS_PIPELINE, 1)
    ctx.reset_accum(); ctx.reset_counters()
    ctx.render_pass(0, n_samples)                       # one call, n_samples passes
    check("n_samples loop")
    ctx.reset_accum(); ctx.reset_counters()
    for s in range(n_samples):                          # other calls in between end and restart the sequence
        ctx.render_pass(s, 1)
        if s % 3 == 1:
            ctx.set_camera(up["camera"])
        if s % 3 == 2:
            ctx.read_output()
    check("interleaved calls")
    ctx.comm_init(ctx.comm_unique_id(), 0, 1)           # a reduce after every pass does not end the sequence
    ctx.reset_accum(); ctx.reset_counters()
    for s in range(n_samples):
        ctx.render_pass(s, 1); ctx.reduce_accum()
    assert np.array_equal(bits(ctx.read_reduced_accum()), bits(ref))
    check("reduce between passes")
    # a view change in the middle of a sequence: the reset lands between the right two passes
    cam2 = rtdx.camera_params((sc.eye[0] + 0.3, sc.eye[1], sc.eye[2]), sc.center, sc.up, W / float(H))
    ctx.reset_accum()
    for s in range(3):
        ctx.render_pass(s, 1)
    ctx.set_camera(cam2)
    for s in range(3, 6):
        ctx.render_pass(s, 1)
    ctx.synchronize()
    ref2 = None
    for s in range(3, 6):
        img, _ = osc.render(cam2, W, H, s, 1, bounces=bounces, flags=0)
        ref2 = img if ref2 is None else ref2 + img
    assert np.array_equal(bits(ctx.read_accum()), bits(ref2))
    ctx.close()


def test_fast_math_pipelined_passes_accumulate_like_unpipelined_ones(rtdx):
    """RTX_FLAG_FAST_MATH with RTX_OPT_PASS_PIPELINE on and off: a run of passes leaves the same accumulation bit for bit.  The passes
    on the caller's stream and those on the two lanes add their samples to gPermanentData with one and the same k_accumulate."""
    sc = rtdx.scenes.mesh_room(n=16)
    W, H, bounces, n_samples = 384, 192, 3, 7
    ctx, _ = _upload(rtdx, sc, W, H, bounces=bounces, flags=rtdx.FLAG_FAST_MATH)
    accs = []
    for pipeline in (1, 0):
        ctx.set_option(rtdx.OPT_PASS_PIPELINE, pipeline)
        ctx.reset_accum()
        for s in range(n_samples):
            ctx.render_pass(s, 1)
        ctx.synchronize()
        accs.append(ctx.read_accum())
    assert (accs[0][..., 3] == n_samples).all()
    assert np.array_equal(bits(accs[0]), bits(accs[1]))
    ctx.close()


def test_last_pass_timing_after_pipelined_and_stage_timed_passes(rtdx):
    """rtx_last_pass_ms / rtx_last_pass_stage_ms.  After a pipelined sequence, whose last pass ran on either lane and carries no
    per-launch events, the pass total is positive and every stage is 0.  With RTX_OPT_STAGE_TIMING the stages are non-negative, the
    closest-hit launches take time, and the stages add up to no more than the pass total."""
    sc = rtdx.scenes.mesh_room(n=16)
    ctx, _ = _upload(rtdx, sc, 384, 192, bounces=3)
    for first, n in ((0, 2), (2, 1)):                   # the sequence goes on across rtx_synchronize: its last pass on lane 1, then lane 0
        for s in range(first, first + n):
            ctx.render_pass(s, 1)
        ctx.synchronize()
        stages, total = ctx.last_pass_stage_ms()
        assert total > 0 and all(v == 0.0 for v in stages.values()), (first, stages, total)
        assert ctx.last_pass_ms() == (0.0, total)
    ctx.set_option(rtdx.OPT_STAGE_TIMING, 1)
    ctx.render_pass(3, 1); ctx.synchronize()
    stages, total = ctx.last_pass_stage_ms()
    assert all(v >= 0.0 for v in stages.values()) and stages["closest"] > 0, stages
    assert sum(stages.values()) <= total + 1e-4, (stages, total)
    assert ctx.last_pass_ms() == (stages["closest"], total)
    ctx.close()


def test_pipelined_frames_are_bit_identical(rtdx, orc):
    """RTX_OPT_FRAME_PIPELINE: a per-frame loop in the reference's order (rtx_set_instances with a moving instance, rtx_set_camera,
    rtx_render_pass, rtx_read_output_async with one frame in flight) on a one-node TLAS keeps two sets of per-frame state and overlaps
    consecutive frames.  The accumulation equals the oracle's frame by frame sum (each sample rendered with that frame's transforms),
    every frame's RGBA8 image equals the one of the same loop with the option off, a camera change in the middle resets the
    accumulation between the right two frames, and calls that leave the pattern (a blocking read, a trace) see the newest state."""
    import torch
    sc = rtdx.scenes.mesh_room(n=16)
    W, H, bounces, n_frames = 384, 192, 2, 8
    base = [np.asarray(i[1], dtype=np.float64).reshape(4, 4).T for i in sc.instances]          # column-vector 4x4
    model_ids = [i[0] for i in sc.instances]
    cam2 = rtdx.camera_params((sc.eye[0] + 0.25, sc.eye[1], sc.eye[2]), sc.center, sc.up, W / float(H))

    def xforms(f):
        out = []
        for k, m in enumerate(base):
            m2 = m.copy()
            if k == 1:
                m2[0, 3] += 0.03 * f; m2[1, 3] += 0.01 * f                                    # the mesh moves, the room (and its light) stays
            out.append(rtdx.xmmatrix_from_colvec(m2))
        return out

    def loop(pipeline, osc=None):
        ctx, up = _upload(rtdx, sc, W, H, bounces=bounces)
        ctx.set_option(rtdx.OPT_FRAME_PIPELINE, pipeline)
        pinned = [torch.empty((H, W, 4), dtype=torch.uint8).pin_memory().numpy() for _ in range(2)]
        images, ref, prev = [], None, up["props"]
        cam = up["camera"]
        for f in range(n_frames):
            props, descs = rtdx.instance_properties(xforms(f), [up["model_ids"][m] for m in model_ids])
            props["prevObjectToWorld"] = prev["objectToWorld"]; props["prevObjectToWorldInverse"] = prev["objectToWorldInverse"]
            props["prevObjectToWorldNormal"] = prev["objectToWorldNormal"]
            prev = props
            ctx.set_instances(descs, props)
            if f == 5:
                cam = cam2.copy()
            ctx.set_camera(cam)
            ctx.render_pass(f, 1)
            if f > 0:
                ctx.wait_output(); images.append(pinned[(f - 1) & 1].copy())
            ctx.read_output_async(pinned[f & 1])
            if osc is not None:
                osc.set_props(props)
                img, _ = osc.render(cam, W, H, f, 1, bounces=bounces, flags=0)
                ref = img if (ref is None or f == 5) else ref + img                            # the view change resets gPermanentData
        ctx.wait_output(); images.append(pinned[(n_frames - 1) & 1].copy())
        accum = ctx.read_accum()                                                               # (leaves the pattern: enter())
        rays = rtdx.scenes.camera_rays(cam, 96, 48)
        hits = ctx.trace(rays)                                                                 # sees the LAST frame's transforms
        ctx.close()
        return images, accum, ref, hits, props

    ctx0, up0 = _upload(rtdx, sc, W, H, bounces=bounces)
    osc = orc.OracleScene(sc, up0["props"], up0["lights"])
    ctx0.close()
    img_on, acc_on, ref, hits_on, last_props = loop(1, osc)
    img_off, acc_off, _, hits_off, _ = loop(0)
    assert np.array_equal(bits(acc_on), bits(ref)) and np.array_equal(bits(acc_off), bits(ref))
    assert len(img_on) == n_frames and all(np.array_equal(a, b) for a, b in zip(img_on, img_off))
    osc.set_props(last_props)
    rays = rtdx.scenes.camera_rays(cam2, 96, 48)
    _assert_hits_equal(hits_on, osc.trace(rays, mode=1)); _assert_hits_equal(hits_off, hits_on)


def test_device_arithmetic_fast_paths_exhaustive(rtdx):
    """csrc/dmath.cuh: the hand-scheduled rsqrt (and shared-reciprocal divide) equal the IEEE operations the oracle defines
    (oracle/det_math.h) on every one of the 2^32 binary32 bit patterns — checked on the device, tolerance 0."""
    ctx = rtdx.Context(16, 16)
    r = ctx.selftest_dmath()
    assert r == {"rsqrt": 0, "div3": 0}, r
    ctx.close()


def test_render_fuzz_hostile_materials_and_lights(rtdx, orc):
    """Shading under hostile inputs, bit-exact against the oracle (E0 and 2 ReSTIR frames): mirror-smooth (Pr = 0, Pr < 0.04),
    over-unity and zero Ks/Kd, the loader's default material (LUT = 0 => Ess = 0 => Inf => 0, ObjLoader.h:415), huge and tiny
    emitters, a zero-area light triangle (normalize(0) = NaN in SampleLightNEE), missing and partly-zero vertex normals."""
    sc = hostile_material_scene(rtdx)
    W, H = 72, 56
    ctx, gpu, cnt, ref, octr = _render_both(rtdx, orc, sc, W, H, 3, 4, rtdx.FLAG_JITTER)
    assert cnt["closest_rays"] == octr["closest_rays"] and cnt["shadow_rays"] == octr["shadow_rays"], (cnt, octr)
    mism = bits(gpu) != bits(ref)
    assert mism.sum() == 0, "radiance mismatches: %d of %d floats" % (mism.sum(), mism.size)
    assert (gpu[..., 3] < 3).any() or np.isfinite(gpu).all()               # non-finite samples are dropped by F20, never stored
    ctx.close()
    _restir_frames(rtdx, orc, sc, W, H, 3, 0, [(None, None)] * 2)


def test_accumulation_reset_on_camera_change(rtdx):
    sc = rtdx.scenes.cornell()
    ctx, up = _upload(rtdx, sc, 64, 64, bounces=2, flags=rtdx.FLAG_LAMBERT_ONLY)
    ctx.render_pass(0, 2)
    a = ctx.read_accum()
    assert a[..., 3].max() == 2.0
    ctx.set_camera(up["camera"])                       # same view: accumulation continues (Pass_spat_di_v7.hlsl:407-423)
    ctx.render_pass(2, 1)
    assert ctx.read_accum()[..., 3].max() == 3.0
    cam2 = rtdx.camera_params((0.2, 1.0, 3.4), sc.center, sc.up, 1.0)
    ctx.set_camera(cam2)                               # view changed by more than s_bias: reset
    ctx.render_pass(0, 1)
    assert ctx.read_accum()[..., 3].max() == 1.0
    ctx.close()


def test_cuda_path_matches_committed_golden_fixtures(rtdx):
    """The CUDA path against tests/golden/golden_kat.json (made by tests/golden/make_golden.py from the oracle) — no oracle
    call at run time."""
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_kat.json")) as f:
        g = json.load(f)["cornell"]
    W = H = g["size"]
    sc = rtdx.scenes.cornell()
    ctx, up = _upload(rtdx, sc, W, H, bounces=2, flags=rtdx.FLAG_JITTER | rtdx.FLAG_LAMBERT_ONLY, samples_per_pass=2)
    ctx.reset_counters()
    ctx.render_pass(0, g["spp"])
    ctx.synchronize()
    acc = ctx.read_accum()
    cnt = ctx.counters()
    assert cnt["closest_rays"] == g["closest_rays"] and cnt["shadow_rays"] == g["shadow_rays"]
    assert [int(v) for v in acc.view(np.uint32).reshape(-1)] == g["accum_bits"]
    hits = ctx.trace(rtdx.scenes.camera_rays(up["camera"], W, H))
    assert [int(v) for v in hits["prim"]] == g["primary_prim"]
    ctx.close()


def test_legacy_cuda_path_matches_committed_golden(rtdx):
    """RTX_FLAG_LEGACY_RR against tests/golden/golden_kat.json["legacy"] — no oracle call at run time."""
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_kat.json")) as f:
        g = json.load(f)["legacy"]
    W = H = g["size"]
    ctx, up = _upload(rtdx, rtdx.scenes.cornell(), W, H, bounces=g["bounces"], flags=rtdx.FLAG_LEGACY_RR, samples_per_pass=4)
    ctx.reset_counters()
    ctx.render_pass(0, g["spp"]); ctx.synchronize()
    cnt = ctx.counters()
    assert cnt["closest_rays"] == g["closest_rays"] and cnt["shadow_rays"] == g["shadow_rays"]
    assert [int(v) for v in ctx.read_accum().view(np.uint32).reshape(-1)] == g["accum_bits"]
    ctx.close()


def test_restir_cuda_path_matches_committed_golden(rtdx):
    """3 ReSTIR frames on the engine against tests/golden/golden_kat.json["restir"] — no oracle call at run time."""
    import json
    import os
    import zlib
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_kat.json")) as f:
        g = json.load(f)["restir"]
    W, H = g["width"], g["height"]
    ctx, up = _upload(rtdx, rtdx.scenes.cornell(), W, H, bounces=g["bounces"], flags=rtdx.FLAG_RESTIR)
    ctx.reset_counters()
    for f in range(g["frames"]):
        ctx.render_frame(f)
    ctx.synchronize()
    cnt = ctx.counters()
    assert cnt["closest_rays"] == g["closest_rays"] and cnt["shadow_rays"] == g["shadow_rays"]
    assert [int(v) for v in ctx.read_accum().view(np.uint32).reshape(-1)] == g["accum_bits"]
    assert int(zlib.crc32(np.ascontiguousarray(ctx.read_restir()).view(np.uint8).tobytes())) == g["reservoir_crc32"]
    ctx.close()


def test_reference_asset_scene_matches_committed_golden(rtdx):
    """The reference's own scene (garage.obj + monke.obj, ingested by this repo's loader into tests/golden/reference_scene.npz)
    on the engine: E0 render, primary hit ids and 3 ReSTIR frames against the oracle's committed outputs — no oracle call."""
    import json
    import os
    import zlib
    from util import load_scene_npz
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    with open(os.path.join(here, "reference_scene_golden.json")) as f:
        g = json.load(f)
    sc = load_scene_npz(rtdx, os.path.join(here, "reference_scene.npz"))
    W, H = g["width"], g["height"]
    ctx, up = _upload(rtdx, sc, W, H, bounces=g["bounces"], flags=rtdx.FLAG_RESTIR)
    ctx.reset_counters()
    ctx.render_pass(0, g["e0"]["spp"]); ctx.synchronize()
    cnt = ctx.counters()
    assert (cnt["closest_rays"], cnt["shadow_rays"]) == (g["e0"]["closest_rays"], g["e0"]["shadow_rays"])
    assert int(zlib.crc32(ctx.read_accum().view(np.uint8).tobytes())) == g["e0"]["accum_crc32"]
    hits = ctx.trace(rtdx.scenes.camera_rays(up["camera"], W, H))
    assert [int(v) for v in hits["inst"]] == g["primary"]["inst"] and [int(v) for v in hits["prim"]] == g["primary"]["prim"]
    ctx.reset_accum(); ctx.reset_counters()
    for f in range(g["restir"]["frames"]):
        ctx.render_frame(f)
    ctx.synchronize()
    cnt = ctx.counters()
    assert (cnt["closest_rays"], cnt["shadow_rays"]) == (g["restir"]["closest_rays"], g["restir"]["shadow_rays"])
    assert int(zlib.crc32(ctx.read_accum().view(np.uint8).tobytes())) == g["restir"]["accum_crc32"]
    assert int(zlib.crc32(np.ascontiguousarray(ctx.read_restir()).view(np.uint8).tobytes())) == g["restir"]["reservoir_crc32"]
    ctx.close()


def test_full_size_properties_c2(rtdx):
    """BASELINE config C2 at full size (1M triangles, 1920x1080, bounces 6): size-independent properties instead of an oracle
    run — determinism (two renders of the same sample are bit-identical), sample counting, ray-count bound 5 + bounces per
    path, any-hit == closest-exists on the primary rays, and linearity of the accumulation (pass 0 + pass 1 == both)."""
    sc = rtdx.scenes.mesh_room(n=296)
    W, H = 1920, 1080
    ctx, up = _upload(rtdx, sc, W, H, bounces=6)
    ctx.reset_counters()
    ctx.render_pass(0, 1); ctx.synchronize()
    a0 = ctx.read_accum(); c0 = ctx.counters()
    assert (a0[..., 3] <= 1).all() and a0[..., 3].mean() > 0.999
    assert c0["paths"] == W * H and c0["closest_rays"] + c0["shadow_rays"] <= c0["paths"] * (5 + 6)
    ctx.reset_accum(); ctx.render_pass(0, 1); ctx.synchronize()
    assert np.array_equal(ctx.read_accum().view(np.uint32), a0.view(np.uint32))            # deterministic
    ctx.render_pass(1, 1); ctx.synchronize()
    a01 = ctx.read_accum()
    ctx.reset_accum(); ctx.render_pass(1, 1); ctx.synchronize()
    a1 = ctx.read_accum()
    assert np.array_equal((a0 + a1).view(np.uint32), a01.view(np.uint32))                  # accumulation is a plain running sum
    for parts in (1, 3, 4):                                                                 # concurrent path ranges (default 2)
        ctx.set_option(rtdx.OPT_PASS_PARTS, parts)
        ctx.reset_accum(); ctx.reset_counters(); ctx.render_pass(0, 1); ctx.synchronize()
        assert np.array_equal(ctx.read_accum().view(np.uint32), a0.view(np.uint32)), parts
        c = ctx.counters()
        assert all(c[k] == c0[k] for k in ("paths", "closest_rays", "shadow_rays")), (parts, c, c0)
    ctx.set_option(rtdx.OPT_PASS_PARTS, 2)
    rays = rtdx.scenes.camera_rays(up["camera"], W, H, step=4)
    ch, ah = ctx.trace(rays), ctx.trace(rays, any_hit=True)
    assert np.array_equal(ch["inst"] != rtdx.MISS, ah["inst"] != rtdx.MISS)
    assert (ch["inst"] != rtdx.MISS).all()                                                  # closed room: every primary ray hits
    img = ctx.read_output()
    assert img.shape == (H, W, 4) and (img[..., 3] == 255).all()
    ctx.close()


def test_full_size_properties_c3(rtdx):
    """BASELINE config C3 at full size (10 M instanced triangles, 1000 instances, 3840x2160, bounces 3, ~0.5 M light triangles):
    size-independent properties — determinism, sample counting, the ray bound 5 + bounces per path, any-hit == closest-exists, and
    invariance of the image under a per-frame TLAS refit with unchanged transforms and under the number of concurrent path ranges."""
    sc = rtdx.scenes.instanced_blobs()
    W, H, bounces = 3840, 2160, 3
    ctx, up = _upload(rtdx, sc, W, H, bounces=bounces)
    assert len(sc.instances) == 1000 and sc.n_triangles() > 10_000_000
    ctx.reset_counters()
    ctx.render_pass(0, 1); ctx.synchronize()
    a0 = ctx.read_accum(); c0 = ctx.counters()
    assert c0["paths"] == W * H and c0["closest_rays"] + c0["shadow_rays"] <= c0["paths"] * (5 + bounces)
    assert (a0[..., 3] <= 1).all() and a0[..., 3].mean() > 0.99 and a0[..., :3].sum() > 0
    ctx.set_instances(up["descs"], up["props"])                       # refit (same transforms): hits must not change
    ctx.set_option(rtdx.OPT_PASS_PARTS, 3)
    ctx.reset_accum(); ctx.reset_counters(); ctx.render_pass(0, 1); ctx.synchronize()
    c1 = ctx.counters()
    assert np.array_equal(ctx.read_accum().view(np.uint32), a0.view(np.uint32))
    assert all(c1[k] == c0[k] for k in ("paths", "closest_rays", "shadow_rays")), (c0, c1)
    rays = rtdx.scenes.camera_rays(up["camera"], W, H, step=8)
    ch, ah = ctx.trace(rays), ctx.trace(rays, any_hit=True)
    assert np.array_equal(ch["inst"] != rtdx.MISS, ah["inst"] != rtdx.MISS)
    hit = ch["inst"] != rtdx.MISS
    assert 0.2 < hit.mean() and (ch["inst"][hit] < 1000).all()
    ctx.close()
