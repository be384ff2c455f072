"""CPU tests (-m "not gpu"): the C++ host mirror of the reference's Renderer slices, the C-ABI library (loads, exports
every declared symbol, refuses to compute without a GPU), and the multi-GPU plumbing on gloo with world_size 2."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from util import host_inputs, load_scene_npz

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- F21 light list, rdn/Renderer.cpp:2123-2233 ------------------------------------------------------------------
def _light_list_numpy(rtdx, sc):
    rows = []
    for ii, (mi, _) in enumerate(sc.instances):
        m = sc.models[mi]
        V = m["vertices"]["position"]; I = m["indices"].reshape(-1, 3)
        ids = sc.material_ids[m["material_id_offset"]: m["material_id_offset"] + I.size].reshape(-1, 3)
        for t in range(I.shape[0]):
            mat = sc.materials[ids[t, 0]]
            ke = mat["Ke"]
            if np.float32(np.float32(ke[0] + ke[1]) + ke[2]) > 0:
                a, b, c = V[I[t, 0]], V[I[t, 1]], V[I[t, 2]]
                area = np.float32(0.5) * np.float32(np.linalg.norm(np.cross((b - a).astype(np.float32), (c - a).astype(np.float32)).astype(np.float32)))
                w = area * np.float32(np.float32(np.float32(ke[0] + ke[1]) + ke[2]) / np.float32(3.0))
                rows.append((a, b, c, ii, w, ke))
    order = sorted(range(len(rows)), key=lambda k: -rows[k][4])     # stable, descending
    return [rows[k] for k in order]


def test_light_list_matches_numpy_restatement(rtdx):
    sc = rtdx.scenes.instanced_blobs(n_models=2, n_side=3, lattice=3, emissive_fraction=0.2)
    lights = rtdx.collect_emissive_triangles(sc)
    ref = _light_list_numpy(rtdx, sc)
    assert len(lights) == len(ref) > 0
    assert (lights["triCount"] == len(ref)).all()
    tot = np.float32(0)
    for r in ref:
        tot = np.float32(tot + r[4])
    assert np.allclose(lights["total_weight"], tot, rtol=1e-5)
    assert np.all(np.diff(lights["weight"]) <= 1e-9)                 # sorted by weight, descending
    assert lights["cdf"][-1] == np.float32(1.0) and np.all(np.diff(lights["cdf"]) >= 0)
    assert np.allclose(lights["weight"].sum(), 1.0, atol=1e-4)
    for k in (0, len(ref) // 2, len(ref) - 1):
        assert lights["instanceID"][k] == ref[k][3] and np.allclose(lights["x"][k], ref[k][0]) and np.allclose(lights["emission"][k], ref[k][5])
        assert np.isclose(lights["weight"][k] * tot, ref[k][4], rtol=1e-4)


def test_light_list_cornell(rtdx):
    sc = rtdx.scenes.cornell()
    lights = rtdx.collect_emissive_triangles(sc)
    assert len(lights) == 2 and (lights["triCount"] == 2).all()
    assert np.allclose(lights["weight"], 0.5) and np.allclose(lights["total_weight"], 2 * 0.125 * 15.0)   # 2 tris of area 0.125, mean Ke 15
    assert (lights["instanceID"] == 0).all()


# ---- F22 instance properties, rdn/Renderer.cpp:2091-2121 + TopLevelASGenerator.cpp:181-199 ---------------------------
def test_instance_properties(rtdx):
    rng = np.random.RandomState(4)
    ms = []
    for _ in range(5):
        A = rng.normal(size=(3, 3)) + 2 * np.eye(3)
        M = np.eye(4); M[:3, :3] = A; M[:3, 3] = rng.normal(size=3) * 3
        ms.append(M)
    props, descs = rtdx.instance_properties([rtdx.xmmatrix_from_colvec(m) for m in ms], [0, 1, 2, 3, 4])
    for k, M in enumerate(ms):
        O = props["objectToWorld"][k].reshape(4, 4).T            # HLSL reading: M[r][c] = mem[4c + r]
        OI = props["objectToWorldInverse"][k].reshape(4, 4).T
        N = props["objectToWorldNormal"][k].reshape(4, 4).T
        assert np.allclose(O, M, atol=1e-6)
        assert np.allclose(OI @ O, np.eye(4), atol=1e-5)
        assert np.allclose(N[:3, :3], np.linalg.inv(M[:3, :3]).T, atol=1e-5)      # inverse-transpose of the upper 3x3
        assert np.allclose(descs["transform"][k], M[:3, :], atol=1e-6)           # 3x4 row-major objectToWorld
        assert descs["instance_id_mask"][k] == (k | (0xFF << 24)) and descs["hit_group_flags"][k] == 2 * k and descs["blas"][k] == k
        assert np.array_equal(props["prevObjectToWorld"][k], props["objectToWorld"][k])


def test_ess_lut_is_deterministic_and_plausible(rtdx):
    m = rtdx.scenes.make_material((.5, .5, .5), roughness=0.5)
    a = m.copy(); b = m.copy()
    rtdx.generate_ess_lut(a, seed=7); rtdx.generate_ess_lut(b, seed=7)
    assert np.array_equal(a["LUT"], b["LUT"])
    lut = a["LUT"][0]
    assert (lut > 0.2).all() and (lut <= 1.0001).all()            # directional albedo of a white GGX lobe


# ---- C ABI ------------------------------------------------------------------------------------------------------
def _declared_symbols(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rtx_[a-z_0-9]+)\s*\(", text)))


def test_abi_library_exports_every_declared_symbol(rtdx):
    lib = rtdx.load_library()
    declared = _declared_symbols("rtx_b200.h")
    assert len(declared) >= 24
    for name in declared:
        assert hasattr(lib, name), "librtx_b200.so does not export %s" % name
    assert sorted(rtdx.ABI_SYMBOLS) == declared
    host = rtdx.load_host_library()
    for name in rtdx.HOST_SYMBOLS:
        assert hasattr(host, name)


def test_python_constants_are_exactly_the_header_flags_and_options(rtdx):
    """include/rtx_b200.h defines exactly these RTX_FLAG_* / RTX_OPT_* names, and each has a Python constant of the same value (the
    bindings of tests and bench)."""
    import re
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "rtx_b200.h")).read()
    defs = dict((m.group(1), int(m.group(2), 0)) for m in re.finditer(r"#define\s+RTX_((?:FLAG|OPT)_\w+)\s+(0x[0-9a-fA-F]+|\d+)u", hdr))
    assert sorted(defs) == sorted(["FLAG_JITTER", "FLAG_LAMBERT_ONLY", "FLAG_RESTIR", "FLAG_LEGACY_RR", "FLAG_FAST_MATH"] + [
        "OPT_TRACE_STATS", "OPT_STAGE_TIMING", "OPT_PASS_PARTS", "OPT_TLAS_REBUILD", "OPT_TRACE_FETCH_TH", "OPT_TRACE_SCHED",
        "OPT_TRACE_WAVES", "OPT_QUEUE_LPT", "OPT_TRACE_CTAS", "OPT_PASS_GRAPH", "OPT_SHADOW_OVERLAP", "OPT_PART_ROWS",
        "OPT_PASS_PIPELINE", "OPT_FRAME_PIPELINE"])
    for name, value in defs.items():
        assert getattr(rtdx, name) == value, name


def test_abi_struct_sizes_match_reference_layouts(rtdx):
    assert rtdx.vertex_dt.itemsize == 28 and rtdx.material_dt.itemsize == 128       # S1, S4
    assert rtdx.props_dt.itemsize == 384 and rtdx.light_dt.itemsize == 80           # S6, S7
    assert rtdx.camera_dt.itemsize == 512 and rtdx.desc_dt.itemsize == 64           # S8, D3D12_RAYTRACING_INSTANCE_DESC
    assert C.sizeof(rtdx.RtxConfig) == 48


def test_no_cpu_fallback(rtdx):
    """Without a CUDA device the product must fail loudly, never fall back to the oracle or any CPU path."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(rtdx.RtxError):
        rtdx.Context(16, 16)
    # argument validation happens before any device work
    lib = rtdx.load_library()
    cfg = rtdx.RtxConfig(0, 0, 16, 16, 3, 4, 4, 0, 1, None)      # wrong struct_size
    h = C.c_void_p()
    assert lib.rtx_create(C.byref(cfg), C.byref(h)) == 1 and b"struct_size" in lib.rtx_last_error()


def test_create_validates_the_path_length_before_touching_a_device(rtdx):
    """ADVICE r1: bounces is bounded by the per-part queue-counter block (E0) and by the legacy estimator's bookkeeping."""
    lib = rtdx.load_library()
    for bounces, flags, ok_arg in ((120, 0, True), (121, 0, False), (61, rtdx.FLAG_LEGACY_RR, False), (60, rtdx.FLAG_LEGACY_RR, True)):
        cfg = rtdx.RtxConfig(C.sizeof(rtdx.RtxConfig), 0, 16, 16, bounces, 4, 4, flags, 1, None)
        h = C.c_void_p()
        st = lib.rtx_create(C.byref(cfg), C.byref(h))
        if h:
            lib.rtx_destroy(h)
        if ok_arg:
            assert st != 1, lib.rtx_last_error()             # passes the argument check (fails later only for want of a GPU)
        else:
            assert st == 1 and b"bounces" in lib.rtx_last_error()


@pytest.mark.parametrize("flag", [4, 64])
def test_create_rejects_unknown_flags_before_touching_a_device(rtdx, flag):
    """A flag bit the engine does not know (4 selected the removed material-binned queues) fails with RTX_ERR_ARG and an error that
    names the valid flags, instead of rendering in some other mode."""
    lib = rtdx.load_library()
    cfg = rtdx.RtxConfig(C.sizeof(rtdx.RtxConfig), 0, 16, 16, 3, 4, 4, rtdx.FLAG_JITTER | flag, 1, None)
    h = C.c_void_p()
    st = lib.rtx_create(C.byref(cfg), C.byref(h))
    if h:
        lib.rtx_destroy(h)
    assert st == 1 and b"unknown flags" in lib.rtx_last_error() and b"RTX_FLAG_FAST_MATH" in lib.rtx_last_error()


def test_engine_free_host_library_has_no_cuda_dependency(rtdx):
    """The CPU arms of bench.py and the scene builders prepare their inputs through librdx_prep.so, which must not pull in the engine."""
    import subprocess
    out = subprocess.run(["ldd", rtdx.HOST_LIB_PATH], capture_output=True, text=True).stdout
    assert "librtx_b200" not in out and "libcuda" not in out and "libcudart" not in out
    out = subprocess.run(["ldd", rtdx.HOST_FULL_LIB_PATH], capture_output=True, text=True).stdout
    assert "librtx_b200" in out                                # the C++ Renderer class does link the engine


def test_product_does_not_reference_the_oracle():
    """The product path may not import, link or call anything under oracle/."""
    pkg = os.path.join(ROOT, "royaltracer-dx_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle/" not in text.replace("oracle/rtx_oracle.cpp tri_test()", "") and "liborc" not in text and "from oracle" not in text, f
    out = subprocess.run(["ldd", os.path.join(pkg, "librtx_b200.so")], capture_output=True, text=True).stdout
    assert "liborc" not in out


# ---- multi-GPU plumbing on gloo, world_size 2 ---------------------------------------------------------------------------
_WORKER = r"""
import os, sys
sys.path.insert(0, %(root)r); sys.path.insert(0, os.path.join(%(root)r, "tests"))
import numpy as np, torch, torch.distributed as dist
import rtdx, importlib
from oracle import orc
from util import host_inputs
rdist = importlib.import_module("royaltracer-dx_b200.dist")
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%(port)d", rank=int(sys.argv[1]), world_size=2)
rank, world = dist.get_rank(), dist.get_world_size()
sc = rtdx.scenes.cornell(); W = H = 16; SPP = 4
props, descs, lights, cam = host_inputs(rtdx, sc, W, H)
osc = orc.OracleScene(sc, props, lights)          # the CPU oracle stands in for the GPU render in this plumbing test
local = torch.zeros(H, W, 4); scratch = torch.zeros(H, W, 4)
for step in range(SPP // world):
    s = rdist.sample_for(step, rank, world)
    acc = local.numpy()
    osc.render(cam, W, H, s, 1, bounces=2, flags=3, accum=acc)
    total = rdist.reduce_accum(local, scratch, dst=0)
if rank == 0:
    np.save(%(out)r, total.numpy())
dist.barrier(); dist.destroy_process_group()
"""


def test_two_rank_sample_partition_and_reduce(rtdx, orc, tmp_path):
    import importlib
    rdist = importlib.import_module("royaltracer-dx_b200.dist")
    assert [rdist.sample_for(s, r, 2) for s in range(2) for r in range(2)] == [0, 1, 2, 3]
    assert rdist.samples_of_rank(7, 1, 2) == [1, 3, 5]
    out = str(tmp_path / "total.npy")
    import socket
    with socket.socket() as so:
        so.bind(("127.0.0.1", 0)); port = so.getsockname()[1]
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % {"root": ROOT, "port": port, "out": out})
    procs = [subprocess.Popen([sys.executable, str(script), str(r)]) for r in range(2)]
    for p in procs:
        assert p.wait(timeout=300) == 0
    total = np.load(out)
    # reference: one process, samples summed per rank in rank-local order, then rank 0 + rank 1 (fp32 sum order of the reduce)
    sc = rtdx.scenes.cornell(); W = H = 16
    props, descs, lights, cam = host_inputs(rtdx, sc, W, H)
    osc = orc.OracleScene(sc, props, lights)
    parts = []
    for r in range(2):
        acc = np.zeros((H, W, 4), dtype=np.float32)
        for s in rdist.samples_of_rank(4, r, 2):
            osc.render(cam, W, H, s, 1, bounces=2, flags=3, accum=acc)
        parts.append(acc)
    assert np.array_equal(total, parts[0] + parts[1])
    # and it equals the 1-GPU image up to fp32 summation order
    one, _ = osc.render(cam, W, H, 0, 4, bounces=2, flags=3)
    assert (total[..., 3] == 4).all() and np.allclose(total, one, rtol=1e-5, atol=1e-6)


# ---- OBJ/MTL ingest (SURVEY.md §8f rank 2; src/Util/ObjLoader.h:393-495) ------------------------------------------------------
OBJ_TEXT = """# synthetic
mtllib t.mtl
o A
v 0 0 0
v 1 0 0
v 1 1 0
v 0 1 0
v 0 0 1
v 2 0 0
v 2 3 0
vn 0 0 1
vn 0 1 0
f 1//1 2//1 3//1
usemtl red
f 1//2 2//2 3//2 4//2
usemtl glow
f -3 -2 -1
usemtl nosuch
f 1 2 5
f 1 6 7 4
"""
MTL_TEXT = """newmtl red
Kd 0.8 0.1 0.1
Ks 0.5 0.5 0.5
d 0.75
Pr 0.4
Pm 1.0
Ps 0.125
Pc 0.25
Ni 1.45
newmtl glow
Kd 1 1 1
Ke 4 5 6
Tr 0.25
Pr 1.0
"""


def test_obj_loader_follows_the_reference_loader(rtdx, tmp_path):
    (tmp_path / "t.obj").write_text(OBJ_TEXT); (tmp_path / "t.mtl").write_text(MTL_TEXT)
    o = rtdx.load_obj(str(tmp_path / "t.obj"), material_offset=5)
    m = o["materials"]
    assert m.size == 3                                              # [default, red, glow]
    assert tuple(m["Kd"][0]) == (1, 1, 1, 1) and tuple(m["Ks"][0]) == (1, 1, 1) and tuple(m["Pr_Pm_Ps_Pc"][0]) == (1, 0, 0, 0)
    assert (m["LUT"][0] == 0).all()                                 # the default material never gets a LUT (ObjLoader.h:415-417)
    assert np.allclose(m["Kd"][1], (0.8, 0.1, 0.1, 0.75)) and np.allclose(m["Pr_Pm_Ps_Pc"][1], (0.4, 1.0, 0.125, 0.25))
    assert m["Ni"][1] == 1.0                                        # Ni is not taken from the MTL (Material ctor, Vertex.h:14-23)
    assert np.allclose(m["Ke"][2], (4, 5, 6)) and np.isclose(m["Kd"][2][3], 0.75)      # Tr = 1 - d
    assert (m["LUT"][1] > 0).all() and (m["LUT"][2] > 0).all()
    # faces: tri (no usemtl -> default), quad (red) split along the shorter diagonal, tri with negative indices (glow),
    # tri with an unknown usemtl (-> default), quad 1 6 7 4 whose diagonal 6-4 is shorter than 1-7
    ids = o["material_ids"].reshape(-1, 3)
    assert (ids[:, 0] == ids[:, 1]).all() and (ids[:, 1] == ids[:, 2]).all()
    assert [int(v) for v in ids[:, 0]] == [5, 6, 6, 7, 5, 5, 5]     # offset 5: default = 5, red = 6, glow = 7
    idx = o["indices"].reshape(-1, 3)
    assert idx.shape[0] == 7
    v = o["vertices"]
    assert v.size == 7                                              # de-duplicated by position only
    assert tuple(v["normal_material"][0][:3]) == (0, 0, 1)          # first normal seen for position 1 wins (Vertex.h:32-34,48)
    p = v["position"][idx]
    assert np.allclose(p[1], [[0, 0, 0], [1, 0, 0], [0, 1, 0]]) and np.allclose(p[2], [[1, 0, 0], [1, 1, 0], [0, 1, 0]])   # unit quad: diag 0-2 == 1-3 -> [0,1,3],[1,2,3]
    assert np.allclose(p[3], [[0, 0, 1], [2, 0, 0], [2, 3, 0]])     # f -3 -2 -1
    assert np.allclose(p[5], [[0, 0, 0], [2, 0, 0], [0, 1, 0]]) and np.allclose(p[6], [[2, 0, 0], [2, 3, 0], [0, 1, 0]])
    assert (v["normal_material"][4][:3] == 0).all()                 # position 5 never had a normal: (0,0,0) (:470-476)
    with pytest.raises(rtdx.RtxError):
        rtdx.load_obj(str(tmp_path / "missing.obj"))


def test_reference_scene_fixture_is_what_the_loader_produces(rtdx):
    """tests/golden/reference_scene.npz = this repo's ingest of the reference's garage.obj + monke.obj.  Where the reference tree
    is mounted (build container) the loader is re-run and compared; everywhere, the known facts of the asset are checked
    (SURVEY.md §2 row 18: 1254 + 967 triangles, 32 emissive triangles with Ke = 5, bbox (-10,-0.055,-5)..(10,4,5))."""
    sc = load_scene_npz(rtdx, os.path.join(ROOT, "tests", "golden", "reference_scene.npz"))
    assert [m["indices"].size // 3 for m in sc.models] == [1254, 967]
    counts = np.bincount(sc.material_ids) // 3
    assert [int(c) for c in counts] == [0, 268, 954, 32, 0, 967]    # [default, black_walls, floor, lights, default, Material.001]
    assert tuple(sc.materials["Ke"][3]) == (5, 5, 5) and rtdx.collect_emissive_triangles(sc).size == 32
    pos = sc.models[0]["vertices"]["position"]
    assert np.allclose(pos.min(0), (-10, -0.054948, -5)) and np.allclose(pos.max(0), (10, 4, 5))
    assert (sc.models[1]["vertices"]["normal_material"][:, :3] == 0).all()      # monke.obj has no normals
    ref_dir = "/root/reference/Pathtracer/include"
    if os.path.exists(os.path.join(ref_dir, "garage.obj")):
        live = rtdx.scenes.reference_scene(ref_dir)
        for a, b in zip(live.models, sc.models):
            assert np.array_equal(a["vertices"], b["vertices"]) and np.array_equal(a["indices"], b["indices"])
        assert np.array_equal(live.material_ids, sc.material_ids) and live.materials.tobytes() == sc.materials.tobytes()
