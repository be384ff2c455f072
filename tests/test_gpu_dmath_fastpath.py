"""-m gpu: the unguarded division / square-root fast paths of the shading stages (csrc/dmath.cuh) and the IEEE replay of the
paths whose operands leave their range (csrc/wavefront.cu k_gi_step)."""
import numpy as np
import pytest

from util import bits, hostile_material_scene

pytestmark = pytest.mark.gpu


def test_fast_paths_exhaustive(rtdx):
    """sqrt, rcp and rsqrt on all 2^32 bit patterns, a / b on 2^34 pairs over every exponent cell of the guard region and one
    binade beyond it, a / 3 and a / pi on every a: each result equals the IEEE operation unless the range flag is raised, and the
    flag is raised exactly outside the stated range."""
    ctx = rtdx.Context(16, 16)
    r = ctx.selftest_dmath_fast_paths()
    assert r == {"sqrt": 0, "rcp": 0, "rsqrt": 0, "div": 0, "div_const": 0}, r
    ctx.close()


def _replays(rtdx, ctx):
    """One pass with the replay counter on; returns (accumulation, counters).  The counting pass runs as one path range."""
    ctx.reset_accum(); ctx.reset_counters(); ctx.set_option(rtdx.OPT_TRACE_STATS, 1)
    ctx.render_pass(0, 1); ctx.synchronize()
    acc, c = ctx.read_accum(), ctx.counters()
    ctx.set_option(rtdx.OPT_TRACE_STATS, 0)
    return acc, c


@pytest.mark.parametrize("config", ["C2", "C3"])
def test_replay_fraction_full_size(rtdx, config):
    """The replayed share of paths at the benchmark's full-size configurations stays below 0.1 %, and counting does not change
    the image."""
    if config == "C2":
        sc, W, H, bounces = rtdx.scenes.mesh_room(n=296, seed=1), 1920, 1080, 8
    else:
        sc, W, H, bounces = rtdx.scenes.instanced_blobs(), 3840, 2160, 3
    ctx = rtdx.Context(W, H, bounces=bounces)
    ctx.upload_scene(sc)
    ctx.render_pass(0, 1); ctx.synchronize()
    a0 = ctx.read_accum()
    acc, c = _replays(rtdx, ctx)
    assert np.array_equal(bits(acc), bits(a0))
    frac = c["shading_replays"] / c["paths"]
    print("%s: %d replayed paths of %d (%.4f %%)" % (config, c["shading_replays"], c["paths"], 100 * frac))
    assert frac < 1e-3, (config, c["shading_replays"], c["paths"])
    ctx.close()


def test_forced_replays_bit_exact(rtdx, orc):
    """A scene whose paths leave the fast paths' range (a zero-area light triangle normalised, the loader's default material with
    Ess = 0, emitters of 1e4 and of 3e-4) replays paths and still matches the oracle bit for bit."""
    sc = hostile_material_scene(rtdx)
    W, H, bounces = 72, 56, 4
    ctx = rtdx.Context(W, H, bounces=bounces, flags=rtdx.FLAG_JITTER)
    up = ctx.upload_scene(sc)
    osc = orc.OracleScene(sc, up["props"], up["lights"])
    gpu, c = _replays(rtdx, ctx)
    ref, _ = osc.render(up["camera"], W, H, 0, 1, bounces=bounces, flags=rtdx.FLAG_JITTER)
    assert c["shading_replays"] > 0
    mism = bits(gpu) != bits(ref)
    assert mism.sum() == 0, "radiance mismatches: %d of %d floats" % (mism.sum(), mism.size)
    ctx.close()
