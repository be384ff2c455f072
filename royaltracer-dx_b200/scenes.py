"""Procedural, seeded scenes for the BASELINE.json configs (SURVEY.md §8d) — synthetic inputs in the reference's
scene description: per model Vertex[] (28 B) + uint32 indices + one material id per face-vertex (global index space,
entry 0 of the material list = the loader's default material, src/Util/ObjLoader.h:415-417), instances as XMMATRIX.
"""
import numpy as np

from . import generate_ess_lut, load_obj, material_dt, ray_dt, vertex_dt, xmmatrix_from_colvec


class SceneDesc:
    def __init__(self):
        self.models = []          # dict(vertices, indices, material_id_offset)
        self.material_ids = np.zeros(0, dtype=np.uint32)
        self.materials = np.zeros(0, dtype=material_dt)
        self.instances = []       # (model index, XMMATRIX memory float32[16])
        self.eye, self.center, self.up = (-1.5, 1.5, 3.5), (0.0, 1.0, 0.0), (0.0, 1.0, 0.0)   # rdn/Renderer.cpp:47-48
        self.name = ""

    def add_model(self, positions, normals, indices, tri_material):
        """positions/normals: (nv,3); indices: (nt,3); tri_material: (nt,) global material index per triangle."""
        nv = positions.shape[0]
        v = np.zeros(nv, dtype=vertex_dt)
        v["position"] = positions.astype(np.float32)
        off = int(self.material_ids.size)
        v["normal_material"][:, :3] = normals.astype(np.float32)
        v["normal_material"][:, 3] = np.float32(off)       # the reference's float smuggling (Hit_v7.hlsl:16-17); the ABI takes the uint
        idx = np.ascontiguousarray(indices.astype(np.uint32).reshape(-1))
        ids = np.repeat(np.asarray(tri_material, dtype=np.uint32), 3)
        self.material_ids = np.concatenate([self.material_ids, ids])
        self.models.append({"vertices": v, "indices": idx, "material_id_offset": off})
        return len(self.models) - 1

    def add_instance(self, model, m4_colvec=None):
        m = np.eye(4, dtype=np.float32) if m4_colvec is None else np.asarray(m4_colvec, dtype=np.float32)
        self.instances.append((model, xmmatrix_from_colvec(m)))

    def n_triangles(self):
        return sum(self.models[i]["indices"].size // 3 for i, _ in self.instances)


def from_obj_files(paths, transforms=None, name="obj"):
    """Renderer::LoadAssets / CreateVB over a model list (rdn/Renderer.cpp:362-370,1973-2072): every OBJ becomes one model
    (one BLAS) with one instance; material blocks and material-id ranges accumulate across models exactly as materialOffset /
    materialVertexOffset do.  transforms: column-vector 4x4 per model (default identity)."""
    sc = SceneDesc(); sc.name = name
    mats = []
    for k, path in enumerate(paths):
        off_mat = sum(m.size for m in mats)
        o = load_obj(path, material_offset=off_mat)
        off_ids = int(sc.material_ids.size)
        v = o["vertices"].copy()
        v["normal_material"][:, 3] = np.float32(off_ids)       # the reference's float smuggling; the ABI takes the uint
        sc.material_ids = np.concatenate([sc.material_ids, o["material_ids"]])
        sc.models.append({"vertices": v, "indices": o["indices"], "material_id_offset": off_ids})
        mats.append(o["materials"])
        sc.add_instance(k, None if transforms is None else transforms[k])
    sc.materials = np.concatenate(mats)
    return sc


def reference_scene(asset_dir):
    """The reference's only scene: garage.obj + monke.obj (rdn/Renderer.cpp:363), instance 1 rotated by 1.57 rad about y every
    frame (:444-449), default camera (:47-48)."""
    import os
    rot = np.eye(4); rot[:3, :3] = _rot_y(np.float32(1.57))        # XMMatrixRotationAxis({0,1,0}, 1.57f), column-vector form
    return from_obj_files([os.path.join(asset_dir, "garage.obj"), os.path.join(asset_dir, "monke.obj")], [np.eye(4), rot],
                          name="garage+monke")


def default_material():
    m = np.zeros(1, dtype=material_dt)
    m["Kd"] = (1, 1, 1, 1); m["Ks"] = (1, 1, 1); m["Ni"] = 1; m["Pr_Pm_Ps_Pc"] = (1, 0, 0, 0)
    return m


def make_material(kd, ks=(0, 0, 0), ke=(0, 0, 0), roughness=1.0, metallic=0.0):
    m = np.zeros(1, dtype=material_dt)
    m["Kd"] = (kd[0], kd[1], kd[2], 1.0); m["Ks"] = ks; m["Ni"] = 1.0; m["Ke"] = ke
    m["Pr_Pm_Ps_Pc"] = (roughness, metallic, 0.0, 0.0)
    return m


def _fill_luts(materials):
    """LUT depends on roughness only: generate once per distinct roughness (fixed seeds), leave the default material at 0."""
    cache = {}
    for i in range(1, len(materials)):
        r = float(materials[i]["Pr_Pm_Ps_Pc"][0])
        if r not in cache:
            one = materials[i:i + 1].copy()
            generate_ess_lut(one, seed=1000 + int(round(r * 1000)))
            cache[r] = one["LUT"][0].copy()
        materials[i]["LUT"] = cache[r]
    return materials


def _quad(p0, p1, p2, p3):
    return [np.array(p, dtype=np.float64) for p in (p0, p1, p2, p3)]


def _box_quads(lo, hi):
    lx, ly, lz = lo; hx, hy, hz = hi
    return [
        _quad((hx, ly, hz), (hx, ly, lz), (hx, hy, lz), (hx, hy, hz)),   # +x
        _quad((lx, ly, lz), (lx, ly, hz), (lx, hy, hz), (lx, hy, lz)),   # -x
        _quad((lx, hy, hz), (hx, hy, hz), (hx, hy, lz), (lx, hy, lz)),   # +y
        _quad((lx, ly, lz), (hx, ly, lz), (hx, ly, hz), (lx, ly, hz)),   # -y
        _quad((lx, ly, hz), (hx, ly, hz), (hx, hy, hz), (lx, hy, hz)),   # +z
        _quad((hx, ly, lz), (lx, ly, lz), (lx, hy, lz), (hx, hy, lz)),   # -z
    ]


def _quads_to_mesh(quads, mats, flip=False):
    pos, idx, tm = [], [], []
    for q, m in zip(quads, mats):
        b = len(pos)
        pos.extend(q)
        if flip:
            idx += [(b, b + 2, b + 1), (b, b + 3, b + 2)]
        else:
            idx += [(b, b + 1, b + 2), (b, b + 2, b + 3)]
        tm += [m, m]
    pos = np.array(pos, dtype=np.float32)
    return pos, np.zeros_like(pos), np.array(idx, dtype=np.uint32), np.array(tm, dtype=np.uint32)


def _rot_y(a):
    c, s = np.cos(a), np.sin(a)
    return np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]])


def cornell():
    """C1: Cornell box, 36 triangles (5 walls x2 + 2 boxes x12 + light x2), flat normals, one model, one instance."""
    sc = SceneDesc(); sc.name = "cornell36"
    WHITE, RED, GREEN, LIGHT = 1, 2, 3, 4
    quads = [
        _quad((-1, 0, 1), (1, 0, 1), (1, 0, -1), (-1, 0, -1)),       # floor  (+y)
        _quad((-1, 2, -1), (1, 2, -1), (1, 2, 1), (-1, 2, 1)),       # ceiling (-y)
        _quad((-1, 0, -1), (1, 0, -1), (1, 2, -1), (-1, 2, -1)),     # back   (+z)
        _quad((-1, 0, 1), (-1, 0, -1), (-1, 2, -1), (-1, 2, 1)),     # left   (+x) red
        _quad((1, 0, -1), (1, 0, 1), (1, 2, 1), (1, 2, -1)),         # right  (-x) green
    ]
    mats = [WHITE, WHITE, WHITE, RED, GREEN]
    for (cx, cz, hw, hh, ang) in [(-0.33, -0.3, 0.3, 1.2, 0.3), (0.35, 0.3, 0.3, 0.6, -0.3)]:
        R = _rot_y(ang)
        for q in _box_quads((-hw, 0.0, -hw), (hw, hh, hw)):
            quads.append([R @ p + np.array([cx, 0.0, cz]) for p in q])
            mats.append(WHITE)
    quads.append(_quad((-0.25, 1.98, -0.25), (0.25, 1.98, -0.25), (0.25, 1.98, 0.25), (-0.25, 1.98, 0.25)))   # light (-y)
    mats.append(LIGHT)
    pos, nrm, idx, tm = _quads_to_mesh(quads, mats)
    assert idx.shape[0] == 36
    sc.materials = np.concatenate([default_material(), make_material((.73, .73, .73)), make_material((.65, .05, .05)),
                                   make_material((.12, .45, .15)), make_material((0, 0, 0), ke=(15, 15, 15))])
    _fill_luts(sc.materials)
    m = sc.add_model(pos, nrm, idx, tm)
    sc.add_instance(m)
    sc.eye, sc.center, sc.up = (0.0, 1.0, 3.4), (0.0, 1.0, 0.0), (0.0, 1.0, 0.0)
    return sc


def _cube_sphere(n, radius, seed, amp):
    """6 x n x n x 2 triangles; sum-of-sines displacement (seeded); smooth area-weighted vertex normals; outward winding."""
    rng = np.random.RandomState(seed)
    t = np.linspace(-1.0, 1.0, n + 1)
    a, b = np.meshgrid(t, t, indexing="ij")
    a = np.tan(a * (np.pi / 4)); b = np.tan(b * (np.pi / 4))       # equal-angle cube map: more uniform triangles
    faces = []
    one = np.ones_like(a)
    for axis in range(3):
        for sgn in (1.0, -1.0):
            c = [None, None, None]
            c[axis] = sgn * one; c[(axis + 1) % 3] = a; c[(axis + 2) % 3] = b
            faces.append(np.stack(c, axis=-1).reshape(-1, 3))
    p = np.concatenate(faces)
    p /= np.linalg.norm(p, axis=1, keepdims=True)
    disp = np.zeros(p.shape[0])
    for k in range(6):
        d = rng.normal(size=3); d /= np.linalg.norm(d)
        f = 2.0 * (1.6 ** k) * (1.0 + rng.rand())
        disp += (0.5 ** k) * np.sin(f * (p @ d) * np.pi + rng.rand() * 6.28)
    p = p * (radius * (1.0 + amp * disp))[:, None]
    ii, jj = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    v00 = (ii * (n + 1) + jj).reshape(-1); v10 = v00 + (n + 1); v01 = v00 + 1; v11 = v10 + 1
    cell = np.concatenate([np.stack([v00, v10, v11], 1), np.stack([v00, v11, v01], 1)])
    idx = np.concatenate([cell + f * (n + 1) * (n + 1) for f in range(6)])
    e1 = p[idx[:, 1]] - p[idx[:, 0]]; e2 = p[idx[:, 2]] - p[idx[:, 0]]
    fn = np.cross(e1, e2)
    cen = (p[idx[:, 0]] + p[idx[:, 1]] + p[idx[:, 2]]) / 3.0
    flip = np.einsum("ij,ij->i", fn, cen) < 0
    idx[flip] = idx[flip][:, [0, 2, 1]]
    fn[flip] *= -1
    vn = np.zeros_like(p)
    for k in range(3):
        np.add.at(vn, idx[:, k], fn)
    ln = np.linalg.norm(vn, axis=1, keepdims=True)
    vn = np.where(ln > 0, vn / np.maximum(ln, 1e-30), 0.0)
    return p.astype(np.float32), vn.astype(np.float32), idx.astype(np.uint32)


def _pbr_materials():
    mats = [default_material()]
    cols = [(.8, .3, .2), (.2, .6, .8), (.7, .7, .2), (.5, .8, .4), (.9, .9, .9), (.4, .3, .7), (.85, .55, .25), (.3, .3, .3)]
    k = 0
    for metallic in (0.0, 1.0):
        for rough in (0.1, 0.3, 0.6, 1.0):
            kd = cols[k]
            ks = kd if metallic else (0.04, 0.04, 0.04)
            mats.append(make_material(kd, ks=ks, roughness=rough, metallic=metallic))
            k += 1
    return mats   # indices 1..8


def mesh_room(n=296, seed=1):
    """C2: displaced cube-sphere with 6*n*n*2 triangles (n=296 -> 1,051,392) inside a 6-quad room with one quad emitter;
    8 PBR materials (roughness {0.1,0.3,0.6,1} x metallic {0,1}) assigned per 16x16-cell patch."""
    sc = SceneDesc(); sc.name = "mesh_room_%d" % (6 * n * n * 2)
    mats = _pbr_materials()
    WALL = len(mats); mats.append(make_material((.7, .7, .7)))
    LIGHT = len(mats); mats.append(make_material((0, 0, 0), ke=(10, 10, 10)))
    sc.materials = _fill_luts(np.concatenate(mats))
    p, vn, idx = _cube_sphere(n, 1.6, seed, 0.06)
    p[:, 1] += 2.0
    nt = idx.shape[0]
    tri = np.arange(nt)
    per_face = n * n * 2
    f = tri // per_face; r = tri % per_face; half = r // (n * n); c = r % (n * n)
    ci, cj = c // n, c % n
    patch = (f * 7 + (ci // 16) * 3 + (cj // 16) * 5 + half * 0) % 8
    m0 = sc.add_model(p, vn, idx, 1 + patch)
    quads = _box_quads((-6.0, 0.0, -6.0), (6.0, 6.0, 6.0))
    wmats = [WALL] * 6
    quads.append(_quad((-2.0, 5.98, -2.0), (2.0, 5.98, -2.0), (2.0, 5.98, 2.0), (-2.0, 5.98, 2.0)))   # emitter, facing -y
    wmats.append(LIGHT)
    pos, nrm, qidx, tm = _quads_to_mesh(quads[:6], wmats[:6], flip=True)       # room walls face inward
    lp, ln_, lidx, ltm = _quads_to_mesh(quads[6:], wmats[6:])
    pos = np.concatenate([pos, lp]); nrm = np.concatenate([nrm, ln_])
    qidx = np.concatenate([qidx, lidx + 24]); tm = np.concatenate([tm, ltm])
    m1 = sc.add_model(pos, nrm, qidx, tm)
    sc.add_instance(m0); sc.add_instance(m1)
    sc.eye, sc.center, sc.up = (-3.5, 3.0, 4.5), (0.0, 2.0, 0.0), (0.0, 1.0, 0.0)
    return sc


def instanced_blobs(n_models=10, n_side=29, lattice=10, emissive_fraction=0.05, seed=3):
    """C3: n_models BLAS of 6*n_side^2*2 (~10k) triangles, lattice^3 instances with seeded TRS; emissive_fraction of the
    instances use a model whose material is an emitter (materials bind per model triangle, so that is one extra BLAS)."""
    sc = SceneDesc(); sc.name = "instanced_%dx%d" % (lattice ** 3, 6 * n_side * n_side * 2)
    mats = _pbr_materials()
    LIGHT = len(mats); mats.append(make_material((0, 0, 0), ke=(6, 5, 4)))
    sc.materials = _fill_luts(np.concatenate(mats))
    rng = np.random.RandomState(seed)
    model_ids = []
    for k in range(n_models):
        p, vn, idx = _cube_sphere(n_side, 0.33, 100 + k, 0.10)
        model_ids.append(sc.add_model(p, vn, idx, np.full(idx.shape[0], 1 + (k % 8))))
    p, vn, idx = _cube_sphere(n_side, 0.33, 100, 0.10)
    emissive_model = sc.add_model(p, vn, idx, np.full(idx.shape[0], LIGHT))
    n_inst = lattice ** 3
    n_em = int(round(n_inst * emissive_fraction))
    order = rng.permutation(n_inst)
    is_em = np.zeros(n_inst, dtype=bool); is_em[order[:n_em]] = True
    k = 0
    for ix in range(lattice):
        for iy in range(lattice):
            for iz in range(lattice):
                i = (ix * lattice + iy) * lattice + iz
                ax = rng.normal(size=3); ax /= np.linalg.norm(ax)
                ang = rng.rand() * 2 * np.pi
                K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
                R = np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * (K @ K)
                s = 0.6 + 0.8 * rng.rand()
                M = np.eye(4); M[:3, :3] = R * s
                M[:3, 3] = np.array([ix, iy, iz]) - (lattice - 1) / 2.0 + (rng.rand(3) - 0.5) * 0.3
                if is_em[i]:
                    sc.add_instance(emissive_model, M)
                else:
                    sc.add_instance(model_ids[k % n_models], M); k += 1
    d = lattice * 0.9
    sc.eye, sc.center, sc.up = (d, d * 0.6, d * 1.1), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0)
    return sc


def sphere_in_box(n_tris_target, seed=5):
    """C5: uniformly tessellated displaced sphere in a box, ~n_tris_target triangles."""
    n = max(2, int(round(np.sqrt(n_tris_target / 12.0))))
    sc = SceneDesc(); sc.name = "sphere_in_box_%d" % (6 * n * n * 2)
    mats = [default_material(), make_material((.7, .7, .7)), make_material((0, 0, 0), ke=(10, 10, 10))]
    sc.materials = _fill_luts(np.concatenate(mats))
    p, vn, idx = _cube_sphere(n, 1.5, seed, 0.05)
    m0 = sc.add_model(p, vn, idx, np.full(idx.shape[0], 1))
    pos, nrm, qidx, tm = _quads_to_mesh(_box_quads((-4, -4, -4), (4, 4, 4)), [1, 1, 2, 1, 1, 1], flip=True)
    m1 = sc.add_model(pos, nrm, qidx, tm)
    sc.add_instance(m0); sc.add_instance(m1)
    sc.eye, sc.center, sc.up = (0.0, 0.0, 3.9), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0)
    return sc


def camera_rays(cam, width, height, step=1):
    """Pinhole primaries exactly as the engine generates them is not needed for trace tests; this numpy version follows the
    closed form of SURVEY.md Appendix C.1 (float32, not bit-identical to the kernels)."""
    viewI = cam["viewI"][0].reshape(4, 4).T      # HLSL matrix: M[r][c] = mem[4c + r]
    projI = cam["projectionI"][0].reshape(4, 4).T
    xs, ys = np.meshgrid(np.arange(0, width, step), np.arange(0, height, step), indexing="xy")
    dx = (xs / width) * 2 - 1; dy = (ys / height) * 2 - 1
    tgt = np.stack([dx, -dy, np.ones_like(dx), np.ones_like(dx)], -1).reshape(-1, 4) @ projI.T
    d = np.concatenate([tgt[:, :3], np.zeros((tgt.shape[0], 1))], 1) @ viewI.T
    d = d[:, :3] / np.linalg.norm(d[:, :3], axis=1, keepdims=True)
    rays = np.zeros(d.shape[0], dtype=ray_dt)
    rays["origin"] = viewI[:3, 3]; rays["direction"] = d.astype(np.float32)
    rays["tmin"] = 1e-4; rays["tmax"] = 1e4
    return rays


def deform(vertices, t, amplitude, seed=0):
    """A seeded, deterministic deformation of a model's vertex array (vertex_dt) for animated-mesh workloads: a travelling wave along
    the vertex normals (amplitude x the model's extent, phase moving with t) plus a twist about a seeded axis through the centre of the
    bounds (amplitude x 1 rad across the extent).  Returns a new float32 vertex_dt array; normals are rotated by the twist, the material
    word is kept.  Vertices without a normal are only twisted."""
    v = np.ascontiguousarray(vertices, dtype=vertex_dt)
    p = v["position"].astype(np.float64)
    n = v["normal_material"][:, :3].astype(np.float64)
    out = v.copy()
    if p.shape[0] == 0:
        return out
    rng = np.random.RandomState(seed)
    k = rng.normal(size=3); k /= np.linalg.norm(k)
    axis = rng.normal(size=3); axis /= np.linalg.norm(axis)
    lo, hi = p.min(axis=0), p.max(axis=0)
    c = 0.5 * (lo + hi)
    size = float((hi - lo).max()) or 1.0
    freq = 2.0 * np.pi * (1.0 + rng.rand()) / size
    phase = 2.0 * np.pi * rng.rand()
    q = p - c
    q = q + n * (amplitude * size * 0.1 * np.sin(freq * (q @ k) - 2.0 * np.pi * t + phase))[:, None]
    ang = amplitude * (q @ axis) / size                     # Rodrigues' rotation about `axis`, angle varying along it
    cs, sn = np.cos(ang)[:, None], np.sin(ang)[:, None]

    def rot(x):
        return x * cs + np.cross(axis, x) * sn + axis * (x @ axis)[:, None] * (1.0 - cs)

    out["position"] = (rot(q) + c).astype(np.float32)
    out["normal_material"][:, :3] = rot(n).astype(np.float32)
    return out
