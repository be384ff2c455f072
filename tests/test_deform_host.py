"""Deforming meshes without a GPU: argument checks of rtx_update_model* that fail before any device work, the oracle side of a model
update, and the seeded deformation the GPU tests and tools/deform_time.py share."""
import ctypes as C

import numpy as np

from deform_util import oracle_update, small_model_scene
from util import compare_hits, host_inputs, random_rays


def test_update_model_with_a_null_context_fails_before_touching_a_device(rtdx):
    lib = rtdx.load_library()
    v = np.zeros(3, dtype=rtdx.vertex_dt)
    for mode in (rtdx.UPDATE_REFIT, rtdx.UPDATE_REBUILD):
        assert lib.rtx_update_model(None, 0, v.ctypes.data_as(C.c_void_p), 3, mode) == 1
        assert b"null context" in lib.rtx_last_error()
        assert lib.rtx_update_model_device(None, 0, None, 0, mode) == 1
        assert b"null context" in lib.rtx_last_error()


def test_deform_is_deterministic_for_a_seed(rtdx):
    v = rtdx.scenes.mesh_room(n=8).models[0]["vertices"]
    a, b = rtdx.scenes.deform(v, 0.25, 0.3, seed=4), rtdx.scenes.deform(v, 0.25, 0.3, seed=4)
    assert a.dtype == rtdx.vertex_dt and a.shape == v.shape
    assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    assert not np.array_equal(a["position"], rtdx.scenes.deform(v, 0.25, 0.3, seed=5)["position"])     # the seed matters
    assert not np.array_equal(a["position"], rtdx.scenes.deform(v, 0.5, 0.3, seed=4)["position"])      # so does the time
    assert np.array_equal(a["normal_material"][:, 3], v["normal_material"][:, 3])                     # the material word is kept
    assert np.abs(a["position"] - v["position"]).max() > 0.05
    still = rtdx.scenes.deform(v, 0.25, 0.0, seed=4)                                                   # amplitude 0: the mesh itself
    assert np.allclose(still["position"], v["position"], atol=1e-6)


def test_oracle_update_traces_the_deformed_mesh(rtdx, orc):
    """The oracle after a model update equals its brute-force definition over the deformed vertices, and differs from the mesh before."""
    for sc in (rtdx.scenes.mesh_room(n=6), small_model_scene(rtdx)):
        props, _, lights, cam = host_inputs(rtdx, sc, 32, 32)
        before = orc.OracleScene(sc, props, lights)
        v = rtdx.scenes.deform(sc.models[0]["vertices"], 0.5, 0.4, seed=2)
        _, osc, _ = oracle_update(orc, sc, props, 0, v, lights=lights)
        rng = np.random.RandomState(3)
        rays = np.concatenate([rtdx.scenes.camera_rays(cam, 32, 32), random_rays(rtdx, rng, 3000, (-2, 0.2, -2), (2, 3.5, 2))])
        ref = osc.trace(rays, mode=0)
        r = compare_hits(osc.trace(rays, mode=1), ref)
        assert r["inst"] == 0 and r["prim"] == 0 and r["t"] == 0 and r["u"] == 0 and r["v"] == 0, r
        assert compare_hits(before.trace(rays, mode=0), ref)["t"] > 0
