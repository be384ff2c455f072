"""The hand-written oracle (oracle/rtx_oracle.cpp) PINNED against the reference's own shader text.

oracle/_ref/libref.so is /root/reference/Pathtracer/shaders/*.hlsl (+ the include/*_v6.hlsl files they #include) compiled for the CPU by
oracle/ref/make_ref.py: a mechanical token filter + oracle/ref/hlsl_shim.h, with TraceRay routed to the oracle's ray caster (the
reference has no source for traversal / intersection) and then into the reference's OWN ClosestHit / Miss / Shadow shaders.  These tests
run RayGen, RayGen2, RayGen3 and the leaf functions of the reference and demand bit-identical results from the oracle:
  F1 RandomFloat, F2 seeds, F3 MapPixelID, F5 ClosestHit, F7-F11 BSDF, F12-F18 samplers + SamplePathSimple, F14 reservoirs, F16 reconnection,
  F19 estimator E0, F20 accumulation + sRGB, and the ReSTIR temporal + spatial passes (SURVEY.md 8f rank 1).
Documented deviations of the oracle from reference undefined behaviour (DESIGN.md D1, D5, D6, D12) are the only differences allowed
and each is asserted to be exactly that deviation.  The library is built where the reference's source tree exists (RTX_REFERENCE_ROOT).

Without the reference the same inputs run through the oracle alone, and every value the comparison covers (under the same masks) must
hash to tests/golden/ref_pins.json.  Those digests were recorded from the oracle at a commit whose pins passed against the reference text
bit for bit; with the reference present they are checked as well.  Each entry also holds digests of up to 32 slices of its first array
along the first axis (image rows, or runs of inputs), so that a mismatch names the rows that differ.  tests/golden/make_ref_pins.py
records them again: it may change a digest only with the whole reference present and no test failing."""
import ctypes as C
import hashlib
import json

import numpy as np
import pytest

from util import bits, hostile_material_scene, host_inputs, load_scene_npz

ref = pytest.importorskip("oracle.ref.ref")

import os
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PINS_PATH = os.path.join(GOLDEN, "ref_pins.json")
RECORD = os.environ.get("RTX_RECORD_REF_PINS") == "1"          # set by tests/golden/make_ref_pins.py
LIVE = ref.available()
REFERENCE_COMPLETE = LIVE and ref.available(6) and ref.legacy_available(2) and ref.legacy_available(12)      # every library a pin uses
needs_reference = pytest.mark.skipif(not LIVE, reason="inspects the reference library itself: needs the reference's source tree "
                                                      "(RTX_REFERENCE_ROOT) or a prebuilt oracle/_ref/libref.so")
with open(PINS_PATH) as _f:
    PINS = json.load(_f)["pins"]
_recorded = {}


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()[:32]


def _slices(a):
    a = np.ascontiguousarray(a)
    return np.array_split(np.arange(a.shape[0]), min(32, a.shape[0])) if a.ndim and a.shape[0] else []


def pin(key, *arrays):
    """The oracle's values that the comparison with the reference covers must be the recorded ones (tests/golden/ref_pins.json)."""
    entry = {"sha256": digest(*arrays), "rows": [digest(arrays[0][r[0]:r[-1] + 1])[:8] for r in _slices(arrays[0])]}
    if RECORD:
        _recorded[key] = entry
        if REFERENCE_COMPLETE:
            return
        # without the reference a recording may only add the slice digests of values that are unchanged
    assert key in PINS, "no recorded reference values for %s (tests/golden/make_ref_pins.py)" % key
    want = PINS[key]
    if want["sha256"] == entry["sha256"]:
        return
    rows = [(int(r[0]), int(r[-1])) for r, a, b in zip(_slices(arrays[0]), want.get("rows", []), entry["rows"]) if a != b]
    where = ("rows %s of %d along the first axis of the values" % (", ".join("%d-%d" % r if r[0] != r[1] else "%d" % r[0] for r in rows),
                                                                    len(arrays[0])) if rows else "what the row digests do not cover (shapes, masks, counts)")
    raise AssertionError("%s: the oracle's values differ from the recorded reference values in %s" % (key, where))


@pytest.fixture(scope="module", autouse=True)
def _write_recorded_pins(request):
    yield
    if RECORD and _recorded and request.session.testsfailed == 0:
        with open(PINS_PATH) as f:
            doc = json.load(f)
        doc["pins"].update(_recorded)
        with open(PINS_PATH, "w") as f:        # one line per check
            f.write('{\n "about": %s,\n "pins": {\n%s\n }\n}\n' % (json.dumps(doc["about"]), ",\n".join(
                "  %s: %s" % (json.dumps(k), json.dumps(v)) for k, v in sorted(doc["pins"].items()))))


def _counts(ctr):
    return np.array([ctr["closest_rays"], ctr["shadow_rays"]], dtype=np.uint64)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@needs_reference
def test_library_is_generated_from_the_reference_defaults():
    cfg = np.zeros(4, dtype=np.uint32)
    ref.lib().ref_config(_p(cfg))
    assert list(cfg) == [3, 4, 4, 1]          # bounces, nee_samples, nee_samples_DI, bsdf_samples_DI (Common_v7.hlsl:8-11)
    from oracle.ref import make_ref
    if os.path.isdir(make_ref.SHADERS):       # the filter touches spellings only: every line of the reference survives, in order
        import difflib
        src = make_ref.expand(make_ref.UNITS["rg1"]).split()
        gen = make_ref.filtered(make_ref.UNITS["rg1"]).split()
        sm = difflib.SequenceMatcher(None, src, gen, autojunk=False)
        assert sm.ratio() > 0.9
        # tokens the filter removed or respelled: nothing but qualifiers, attributes, literals' suffixes, swizzle calls, references
        touched = [t for tag, i1, i2, j1, j2 in sm.get_opcodes() if tag != "equal" for t in src[i1:i2]]
        assert len(touched) < 0.12 * len(src)


def test_rng_seeds_and_pixel_map_equal_the_reference(orc):
    L, O = ref.lib() if LIVE else None, orc.lib()
    rng = np.random.RandomState(1)
    outs, seeds, pixels = [], [], []
    for sx, sy in [(0, 0), (1, 2), (0xFFFFFFFF, 0x9e3779b9)] + [tuple(int(v) for v in rng.randint(0, 2 ** 32, size=2, dtype=np.uint64)) for _ in range(200)]:
        b = np.zeros(500, dtype=np.float32); sb = np.zeros(2, dtype=np.uint32)
        O.orc_kat_rng(sx, sy, 500, _p(b), _p(sb))
        if L:
            a, sa = ref.kat_rng(sx, sy, 500)
            assert np.array_equal(bits(a), bits(b)) and np.array_equal(sa, sb)
        outs.append(bits(b)); seeds.append(sb)
    for w, h in [(1920, 1080), (37, 23), (4, 4), (5, 9)]:
        for _ in range(3000):
            x, y = int(rng.randint(0, w)), int(rng.randint(0, h))
            o = O.orc_kat_map_pixel(w, h, x, y)
            if L:
                assert L.ref_kat_map_pixel(w, h, x, y) == o
            pixels.append(o)
    pin("rng", np.array(outs), np.array(seeds))
    pin("map_pixel", np.array(pixels, dtype=np.uint32))


def test_bsdf_functions_equal_the_reference(rtdx, orc):
    """EvaluateBRDF / BRDF_PDF (both lobes), CalculateStrategyProbabilities, SampleBRDF (both), SelectSamplingStrategy on every material
    class of the bench scene (fp16 MaterialOptimized, GGX roughness 0.1..1, metallic 0/1, the LUT-less default material)."""
    sc = rtdx.scenes.mesh_room(n=4)
    props, descs, lights, cam = host_inputs(rtdx, sc, 8, 8)
    osc = orc.OracleScene(sc, props, lights)
    rs = ref.RefScene(sc, props, lights, osc) if LIVE else None
    L, O = ref.lib() if LIVE else None, orc.lib()
    rng = np.random.RandomState(2)
    n_mat = len(sc.materials)

    def unit(v):
        return (v / np.linalg.norm(v)).astype(np.float32)
    bad = {}
    N = 6000
    outs = [[] for _ in range(8)]
    for k in range(N):
        n, i, o = unit(rng.normal(size=3)), unit(rng.normal(size=3)), unit(rng.normal(size=3))
        if k % 3 == 0:
            o = unit(n + 0.3 * rng.normal(size=3)); i = unit(-n + 0.3 * rng.normal(size=3))   # the common configuration
        if k % 7 == 0:
            o = (o * rng.uniform(0.1, 4.0)).astype(np.float32)                                   # un-normalised outgoing (pdf paths)
        mat = int(rng.randint(0, n_mat + 1))                                                    # n_mat = out of bounds -> zeros
        for op in range(8):
            seed = rng.randint(0, 2 ** 32, size=2, dtype=np.uint64).astype(np.uint32)
            sa, sb = seed.copy(), seed.copy()
            a = np.zeros(4, dtype=np.float32); b = np.zeros(4, dtype=np.float32)
            O.orc_kat_bsdf(osc.h, op, mat, _p(n), _p(i), _p(o), _p(sb), _p(b))
            outs[op].append(np.concatenate([bits(b + 0), sb]))                                 # + 0: -0 == +0
            if L:
                L.ref_kat_bsdf(op, mat, _p(n), _p(i), _p(o), _p(sa), _p(a))
                if not (np.array_equal(bits(a + 0), bits(b + 0)) and np.array_equal(sa, sb)):
                    bad[op] = bad.get(op, 0) + 1
    assert not bad, "ops differing from the reference (of %d inputs each): %s" % (N, bad)
    for op in range(8):
        pin("bsdf/op%d" % op, np.array(outs[op]))


def test_bsdf_functions_equal_the_reference_on_hostile_inputs(rtdx, orc):
    """The same eight BSDF entry points with zero, negative-zero, denormal, huge, infinite and NaN components in the normal, incidence and
    outgoing vectors (a quarter of all components): every result equals the reference text's bit for bit (a NaN equals any NaN)."""
    sc = rtdx.scenes.mesh_room(n=4)
    props, descs, lights, cam = host_inputs(rtdx, sc, 8, 8)
    osc = orc.OracleScene(sc, props, lights)
    rs = ref.RefScene(sc, props, lights, osc) if LIVE else None
    L, O = ref.lib() if LIVE else None, orc.lib()
    n_mat = len(sc.materials)
    specials = [0.0, -0.0, 1.0, -1.0, 1e-30, -1e-30, 1e30, np.inf, -np.inf, np.nan, 1e-45, 0.5, 3.4e38]
    rng = np.random.RandomState(5)

    def vec():
        v = rng.normal(size=3).astype(np.float32)
        v /= np.linalg.norm(v)
        for c in range(3):
            if rng.rand() < 0.25:
                v[c] = np.float32(specials[rng.randint(len(specials))])
        return v
    bad = {}
    outs = [[] for _ in range(8)]
    for k in range(4000):
        n, i, o = vec(), vec(), vec()
        mat = int(rng.randint(0, n_mat + 1))
        for op in range(8):
            seed = rng.randint(0, 2 ** 32, size=2, dtype=np.uint64).astype(np.uint32)
            sa, sb = seed.copy(), seed.copy()
            a = np.zeros(4, dtype=np.float32); b = np.zeros(4, dtype=np.float32)
            O.orc_kat_bsdf(osc.h, op, mat, _p(n), _p(i), _p(o), _p(sb), _p(b))
            outs[op].append(np.concatenate([bits(np.where(np.isnan(b), np.float32(np.nan), b + 0)), sb]))     # one NaN for every NaN
            if L:
                L.ref_kat_bsdf(op, mat, _p(n), _p(i), _p(o), _p(sa), _p(a))
                same = np.array_equal(sa, sb) and all((np.isnan(x) and np.isnan(y)) or bits(np.float32(x) + 0) == bits(np.float32(y) + 0) for x, y in zip(a, b))
                if not same:
                    bad[op] = bad.get(op, 0) + 1
    assert not bad, bad
    for op in range(8):
        pin("bsdf_hostile/op%d" % op, np.array(outs[op]))


@needs_reference
def test_reservoir_updates_equal_the_reference(orc):
    """UpdateReservoir / UpdateReservoir_GI (Reservoir_v7.hlsl:30-80) through the pass-1 comparison below; here the uint16 M arithmetic."""
    L = ref.lib()
    rng = np.random.RandomState(3)
    for gi in (0, 1):
        for _ in range(2000):
            w = np.array([rng.uniform(0, 5)], dtype=np.float32); M = np.array([float(rng.randint(0, 200))], dtype=np.float32)
            wi, M_in = float(np.float32(rng.uniform(0, 3))), float(rng.randint(0, 130))
            seed = rng.randint(0, 2 ** 32, size=2, dtype=np.uint64).astype(np.uint32)
            u, _ = ref.kat_rng(int(seed[0]), int(seed[1]), 1)
            w0, M0 = w.copy(), M.copy()
            acc = L.ref_kat_update_reservoir(gi, _p(w), _p(M), wi, M_in, _p(seed))
            assert bits(w)[0] == bits(np.float32(w0[0] + np.float32(wi)))[0] and M[0] == float((int(M0[0]) + int(M_in)) & 0xFFFF)
            assert acc == int(u[0] < np.float32(wi) / w[0])


SCENES = {
    "mesh_room": lambda rtdx: rtdx.scenes.mesh_room(n=8),                                  # closed room, GGX + diffuse, two instances
    "garage_monke": lambda rtdx: load_scene_npz(rtdx, os.path.join(GOLDEN, "reference_scene.npz")),   # the reference's own assets
    "cornell": lambda rtdx: rtdx.scenes.cornell(),                                         # open front: primary misses (deviation D1)
    "hostile_materials": hostile_material_scene,                                           # Pr = 0, Ks > 1, LUT = 0, zero-area light, missing normals
    "instanced_emitters": lambda rtdx: rtdx.scenes.instanced_blobs(n_models=2, n_side=5, lattice=3, emissive_fraction=0.15),   # 27 instances, many lights, open
}
OPEN_SCENES = ("cornell", "instanced_emitters")                                            # primary rays can miss (deviation D1)


def _primary_miss_mask(orc, osc, cam, W, H, sample, bounces):
    m = np.zeros((H, W), dtype=bool)
    for y in range(H):
        for x in range(W):
            m[y, x] = orc.unpack_debug(osc.debug_pixel(cam, W, H, x, y, sample, bounces=bounces))["hit_inst"][0] == 0xFFFFFFFF
    return m


@pytest.mark.parametrize("name", sorted(SCENES))
@pytest.mark.parametrize("bounces", [3, 6])
def test_pass1_and_estimator_e0_equal_the_reference(rtdx, orc, name, bounces):
    """RayGen (Pass_init_di_v7.hlsl:48-190) run from the reference's text per pixel, then E0 (F19) from the reference's ReconnectDI /
    GetP_Hat_GI on its reservoirs: the oracle's accumulation of the same sample is bit-identical on every pixel whose primary ray hits.
    bounces = 6 is BASELINE config C2's path length (the reference's `#define bounces 3` set to 6 in the generated copy)."""
    live = ref.available(None if bounces == 3 else bounces)
    W, H = 48, 32
    sc = SCENES[name](rtdx)
    props, descs, lights, cam = host_inputs(rtdx, sc, W, H)
    osc = orc.OracleScene(sc, props, lights)
    rs = ref.RefScene(sc, props, lights, osc, bounces=None if bounces == 3 else bounces) if live else None
    if rs:
        rs.frame(W, H)
    for sample in (0, 11):
        acc, ctr = osc.render(cam, W, H, sample, 1, bounces=bounces)
        miss = _primary_miss_mask(orc, osc, cam, W, H, sample, bounces)
        if name not in OPEN_SCENES:
            assert not miss.any()
        assert (acc[..., 3] == 1).all()
        # without the reference the oracle's ray counts are pinned exactly (the reference's own counts are bounded below)
        pin("pass1/%s/b%d/s%d" % (name, bounces, sample), bits(np.where(miss[..., None], 0, acc[..., :3])), miss, _counts(ctr))
        if not rs:
            continue
        rs.set_camera(cam, sample)
        rs.dispatch(1)
        e0 = rs.e0()
        rc, rsh = rs.ray_counts()
        differ = (bits(e0[..., :3] + 0) != bits(acc[..., :3])).any(-1)
        assert not (differ & ~miss).any(), "%d pixels differ from the reference" % int((differ & ~miss).sum())
        if not miss.any():
            # ray counts: the oracle issues the reference's rays minus the visibility rays whose result cannot matter (deviation D6)
            # (with the hostile materials most candidates have no contribution at all: most visibility rays are skipped)
            # and more paths end on emitters without contribution, where the reference traces on for nothing: deviation D4)
            slack, slack_c = (2.0, 1.03) if name == "hostile_materials" else (1.2, 1.01)
            assert ctr["closest_rays"] <= rc <= ctr["closest_rays"] * slack_c + 4 and ctr["shadow_rays"] <= rsh <= ctr["shadow_rays"] * slack + 8


def _frames(rtdx, orc, key, sc, W, H, script, allow_miss=False):
    """The reference's frame loop (rdn/Renderer.cpp:431-452,611-673) on both sides: per frame OnUpdate (camera with prevView /
    prevProjection, instance matrices with prev*), then RayGen, RayGen2, RayGen3."""
    props, descs, lights, cam = host_inputs(rtdx, sc, W, H)
    osc = orc.OracleScene(sc, props, lights)
    rs = ref.RefScene(sc, props, lights, osc) if LIVE else None
    if rs:
        rs.frame(W, H)
    frames = osc.new_frames(W, H)
    acc = np.zeros((H, W, 4), dtype=np.float32)
    model_ids = [i[0] for i in sc.instances]
    prev_props = props
    worst = 0
    for f, (new_cam, xforms) in enumerate(script):
        if xforms is not None:
            props, _ = rtdx.instance_properties(xforms, model_ids)
            if f > 0:
                for k in ("objectToWorld", "objectToWorldInverse", "objectToWorldNormal"):
                    props["prev" + k[0].upper() + k[1:]] = prev_props[k]
            osc.set_props(props)
            if rs:
                rs.set_props(props)
            prev_props = props
        if new_cam is not None:
            new_cam = new_cam.copy()
            new_cam["prevView"] = cam["view"]; new_cam["prevProjection"] = cam["projection"]
            cam = new_cam
        elif f > 0:
            cam = cam.copy(); cam["prevView"] = cam["view"]; cam["prevProjection"] = cam["projection"]
        view_changed = np.abs(cam["view"] - cam["prevView"]).max() > 2e-5
        if view_changed:
            acc[:] = 0                                   # the oracle's host-side form of Pass_spat_di_v7.hlsl:407-423
        osc.render_frame(cam, W, H, f, frames, acc, bounces=3)
        b = osc.dump_frames(frames, W, H)
        kind = b[..., 35].copy(); b[..., 35] = 0         # oracle-internal tag: 0 primary miss, 2 sampled, 3 emitter
        sampled = (kind == 2)[..., None]
        pin("%s/frame%d" % (key, f), bits(np.where((kind != 0)[..., None], b, 0) if allow_miss else b), kind,
            bits(np.where(sampled, acc + 0, 0)), np.where(sampled, orc.resolve(acc)[..., :3], 0) if not view_changed else np.zeros(0))
        if not rs:
            continue
        rs.set_camera(cam, f)
        for p in (1, 2, 3):
            rs.dispatch(p)
        a = rs.dump(last=True)
        differ = (bits(a) != bits(b)).any(-1)
        if allow_miss:
            assert not (differ & (kind != 0)).any(), "frame %d: %d non-miss pixels differ" % (f, int((differ & (kind != 0)).sum()))
        else:
            assert not differ.any(), "frame %d: %d pixels' reservoirs / samples differ from the reference" % (f, int(differ.sum()))
        # accumulation (F20): identical except where the primary hit is an emitter (deviation D5: the reference bypasses gPermanentData)
        pm = rs.permanent()
        dacc = (bits(pm + 0) != bits(acc + 0)).any(-1)       # + 0: the first frame stores -0 as it is, the oracle's running sum holds +0
        assert not (dacc & (kind == 2)).any(), "frame %d: accumulation differs on %d sampled pixels" % (f, int((dacc & (kind == 2)).sum()))
        assert (pm[kind == 3] == 0).all()
        # output (sRGB -> UNORM8) on the sampled pixels.  On the frame of a view change the reference displays the average that still
        # contains the stale history (averagedColor is computed at :405 BEFORE the reset at :407-423); gPermanentData, compared above, is
        # identical after the frame (DESIGN.md deviation D14), so the images agree again from the next frame on.
        if view_changed:
            continue
        out = np.zeros((H, W, 4), dtype=np.float32); rs.L.ref_read_output(_p(out))
        u8 = (np.clip(out[..., :3], 0, 1) * np.float32(255.0) + np.float32(0.5)).astype(np.int32)
        assert np.array_equal(u8[kind == 2], orc.resolve(acc)[..., :3].astype(np.int32)[kind == 2])
        worst = max(worst, int(differ.sum()))
    osc.free_frames(frames)
    return worst


def test_restir_frames_static_equal_the_reference(rtdx, orc):
    """RayGen + RayGen2 (temporal) + RayGen3 (spatial, shade, accumulate, sRGB) from the reference's text, 4 frames."""
    _frames(rtdx, orc, "restir_static/mesh_room", SCENES["mesh_room"](rtdx), 48, 32, [(None, None)] * 4)
    _frames(rtdx, orc, "restir_static/cornell", SCENES["cornell"](rtdx), 40, 32, [(None, None)] * 3, allow_miss=True)
    _frames(rtdx, orc, "restir_static/hostile_materials", SCENES["hostile_materials"](rtdx), 40, 30, [(None, None)] * 3)          # reuse across NaN-prone materials and a zero-area light


def test_restir_frames_reference_scene_with_rotating_instance_equal_the_reference(rtdx, orc):
    """garage.obj + monke.obj, instance 1 = rotY(1.57 * frame) as rdn/Renderer.cpp:444-449 animates it, default camera."""
    sc = SCENES["garage_monke"](rtdx)
    base = [np.asarray(i[1], dtype=np.float64).reshape(4, 4).T for i in sc.instances]

    def at(t):
        a = np.float32(1.57) * t
        R = np.eye(4); R[0, 0] = np.cos(a); R[0, 2] = np.sin(a); R[2, 0] = -np.sin(a); R[2, 2] = np.cos(a)
        return [rtdx.xmmatrix_from_colvec(base[0]), rtdx.xmmatrix_from_colvec(R)]
    _frames(rtdx, orc, "restir_rotating_instance", sc, 48, 32, [(None, at(0.0)), (None, at(0.02)), (None, at(0.04)), (None, None)])


def test_restir_frames_moving_camera_equal_the_reference(rtdx, orc):
    sc = SCENES["mesh_room"](rtdx)
    W, H = 40, 32
    cams = [None, rtdx.camera_params((sc.eye[0] + 0.05, sc.eye[1], sc.eye[2]), sc.center, sc.up, W / H),
            rtdx.camera_params((sc.eye[0] + 0.10, sc.eye[1] + 0.02, sc.eye[2]), sc.center, sc.up, W / H), None]
    _frames(rtdx, orc, "restir_moving_camera", sc, W, H, [(c, None) for c in cams])


# ---- the reference's first estimator (SURVEY.md 8f rank 4): include/RayGen.hlsl + include/Hit.hlsl + include/Miss.hlsl -----------------
@pytest.mark.parametrize("name", sorted(SCENES))
@pytest.mark.parametrize("bounces", [2, 12])
def test_legacy_estimator_equals_the_reference_text(rtdx, orc, name, bounces):
    """RayGen (include/RayGen.hlsl:48-187: jittered camera ray, path loop, Russian roulette after depth 3, accumulation) and ClosestHit
    (include/Hit.hlsl:59-357: face-forwarded normals, RIS over 10 light candidates, the nested shadow TraceRay, BSDF sample, MIS on
    emitter hits) run from the reference's own text, one DispatchRays per sample: gPermanentData and the closest / shadow ray counts of
    the oracle's `legacy` estimator (what RTX_FLAG_LEGACY_RR is tested against) are bit-identical on every pixel, for one sample and
    accumulated over three.  The only edit to the text is RayGen.hlsl:63's `uint bounces = 10000000` -> the cap under test (D13);
    the legacy text's older Material / InstanceProperties / LightTriangle layouts are filled field by field (ref_legacy_harness.cpp)."""
    live = ref.legacy_available(bounces)
    from oracle.ref import make_ref
    if os.path.isdir(make_ref.INCLUDE) and name == "cornell":      # the filter touches spellings only, here too
        import difflib
        for unit in ("leg_rg", "leg_hit"):
            src = make_ref.expand(make_ref.LEGACY_UNITS[unit]).split()
            gen = make_ref.filtered_legacy(make_ref.LEGACY_UNITS[unit], bounces).split()
            sm = difflib.SequenceMatcher(None, src, gen, autojunk=False)
            touched = [t for tag, i1, i2, j1, j2 in sm.get_opcodes() if tag != "equal" for t in src[i1:i2]]
            assert sm.ratio() > 0.9 and len(touched) < 0.12 * len(src), (unit, sm.ratio(), len(touched), len(src))
    W, H = 40, 24
    sc = SCENES[name](rtdx)
    props, descs, lights, cam = host_inputs(rtdx, sc, W, H)
    osc = orc.OracleScene(sc, props, lights)
    rs = ref.RefScene(sc, props, lights, osc, bounces=bounces, legacy=True) if live else None
    if rs:
        cfg = np.zeros(4, dtype=np.uint32)
        rs.L.ref_config(_p(cfg))
        assert cfg[0] == 10                                               # RIS_M (include/Common.hlsl:8)
        rs.frame(W, H)
        rs.ray_counts()                                                   # (the library is shared between tests: start the counters at zero)
    flags = orc.FLAG_LEGACY_RR | orc.FLAG_JITTER                          # RayGen.hlsl:86-87 always jitters
    zeros = np.zeros((H, W, 4), dtype=np.float32)
    for sample in (0, 5):
        b, ctr = osc.render(cam, W, H, sample, 1, bounces=bounces, flags=flags)
        assert np.isfinite(b).all() and b[..., :3].sum() > 0 and ((b[..., 3] == 1).all() or name == "hostile_materials")   # (non-finite samples are dropped: RayGen.hlsl:145)
        pin("legacy/%s/b%d/s%d" % (name, bounces, sample), bits(b + 0), _counts(ctr))
        if rs:
            rs.L.ref_write_permanent(_p(zeros))
            rs.set_camera(cam, sample)
            rs.dispatch(1)
            a, rc = rs.permanent(), rs.ray_counts()
            assert rc == (ctr["closest_rays"], ctr["shadow_rays"]), (sample, rc, ctr)
            assert np.array_equal(bits(a + 0), bits(b + 0)), (sample, int((bits(a + 0) != bits(b + 0)).any(axis=2).sum()))
    # three samples accumulated by the reference's own temporal accumulation (RayGen.hlsl:140-156), then its averaged output (:176-183)
    b, _ = osc.render(cam, W, H, 0, 3, bounces=bounces, flags=flags)
    pin("legacy/%s/b%d/accum3" % (name, bounces), bits(b + 0))
    if not rs:
        return
    rs.L.ref_write_permanent(_p(zeros))
    for sample in range(3):
        rs.set_camera(cam, sample)
        rs.dispatch(1)
    a = rs.permanent()
    assert np.array_equal(bits(a + 0), bits(b + 0))
    # The legacy RayGen displays sum / max(count BEFORE this frame, 1) (RayGen.hlsl:142,176-177: frameCount is read before the
    # accumulation): its third frame shows the three-sample sum over 2.  The engine resolves every accumulation buffer with the current
    # count (F20, Common_v7 / Pass_spat_di_v7.hlsl:425-444); only gPermanentData is the legacy row's contract.  Asserted as found:
    out = rs.output()
    if name != "hostile_materials":        # (there the count before the frame differs per pixel: dropped samples)
        assert np.array_equal(bits(out[..., :3] + 0), bits((b[..., :3] / np.float32(2.0)) + 0))
