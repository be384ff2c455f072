"""Helpers of the deforming-mesh tests: the same scene with one model's vertices replaced, on the oracle side and on the engine side."""
import copy

import numpy as np


def with_vertices(scene, model, vertices):
    """A shallow copy of a scenes.SceneDesc whose model `model` has the given vertices (same indices, same material offset)."""
    sc = copy.copy(scene)
    sc.models = list(scene.models)
    sc.models[model] = dict(scene.models[model], vertices=np.ascontiguousarray(vertices))
    return sc


def oracle_update(orc, scene, props, model, vertices, lights=None, rtdx=None):
    """The oracle after a model's positions and normals changed: a scene over the new vertices with its BVH2 built from them (the
    oracle's scene is immutable; rendering state — accumulation, ReSTIR frames — lives outside it and carries over).  The light list is
    the given one, or collected again from the new vertices when rtdx is given.  Returns (new scene desc, oracle scene, lights)."""
    sc = with_vertices(scene, model, vertices)
    if lights is None:
        lights = rtdx.collect_emissive_triangles(sc)
    return sc, orc.OracleScene(sc, props, lights), lights


def small_model_scene(rtdx):
    """A model of 6 triangles (a tetrahedron on a quad: a single-node BLAS) inside a room with an emitter."""
    sc = rtdx.scenes.SceneDesc(); sc.name = "small"
    sc.materials = rtdx.scenes._fill_luts(np.concatenate([rtdx.scenes.default_material(), rtdx.scenes.make_material((.7, .6, .5)),
                                                          rtdx.scenes.make_material((.6, .6, .6)),
                                                          rtdx.scenes.make_material((0, 0, 0), ke=(8, 8, 8))]))
    p = np.array([[-0.5, 0.5, -0.4], [0.5, 0.5, -0.4], [0.0, 0.5, 0.5], [0.0, 1.3, 0.0],
                  [-1.0, 0.3, -1.0], [1.0, 0.3, -1.0], [1.0, 0.3, 1.0], [-1.0, 0.3, 1.0]], dtype=np.float32)
    n = p - p.mean(axis=0); n /= np.linalg.norm(n, axis=1, keepdims=True)
    idx = np.array([[0, 2, 1], [0, 1, 3], [1, 2, 3], [2, 0, 3], [4, 6, 5], [4, 7, 6]])
    m0 = sc.add_model(p, n.astype(np.float32), idx, np.full(6, 1))
    pos, nrm, qidx, tm = rtdx.scenes._quads_to_mesh(rtdx.scenes._box_quads((-3.0, 0.0, -3.0), (3.0, 3.0, 3.0)), [2] * 6, flip=True)
    lq = [rtdx.scenes._quad((-0.7, 2.98, -0.7), (0.7, 2.98, -0.7), (0.7, 2.98, 0.7), (-0.7, 2.98, 0.7))]      # emitter facing -y
    lp, ln_, lidx, ltm = rtdx.scenes._quads_to_mesh(lq, [3])
    m1 = sc.add_model(np.concatenate([pos, lp]), np.concatenate([nrm, ln_]), np.concatenate([qidx, lidx + 24]), np.concatenate([tm, ltm]))
    sc.add_instance(m0); sc.add_instance(m1)
    sc.eye, sc.center, sc.up = (0.5, 1.4, 2.6), (0.0, 0.7, 0.0), (0.0, 1.0, 0.0)
    return sc
