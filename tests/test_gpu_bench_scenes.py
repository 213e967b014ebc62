"""Parity on the scenes that bench.py actually times (VERDICT r1 weak #1) and on the tile-shard hand-off (weak #2).

The four `bench.make_scene` workloads -- C1 Cornell + 868,480 triangles, C2 material room, C3 12.5 M flattened
instance triangles, C4 650,000 curve segments -- are built with the SAME generator arguments as bench.py (same
geometry, BVH, light tables, top-level cut, 32 Ki-bin ray sort) and rendered at reduced resolution / spp so that the
CPU oracle finishes in seconds; the CUDA path is compared with the oracle (pixels and the full hit record of 200 k
random rays) through the C ABI.  Bars are per scene, <= 3x what was measured when the test was written
(the measured value is printed by every run).
"""
import os

import numpy as np
import pytest

from tungsten_b200 import scene, synth, lib, integrator, abi
from oracle import pyoracle

pytestmark = pytest.mark.gpu

RES = (240, 136)          # 15 x 9 tiles (8.5 rows: ragged last row)


def _build(config, d, res=RES, spp=2):
    """Same generator calls as bench.make_scene (bench.py), different resolution."""
    if config == "c1":
        return synth.cornell_dragon_standin(d, res=res, spp=spp)
    if config == "c2":
        synth.save_rgbe(os.path.join(d, "room_env.hdr"), synth.sky_envmap(512, 256))
        return synth.material_room(d, "room", res=res, spp=spp, max_bounces=16, subdiv=6, env="room_env.hdr")
    if config == "c3":
        return synth.instanced_forest(d, "forest10m", n_instances=490, tree_subdiv=5, res=res, spp=spp, extent=40.0)
    if config == "c4":
        return synth.hair_scene(d, "hair650k", n_curves=10000, nodes_per_curve=67, res=res, spp=spp, width=0.004)
    raise KeyError(config)


def _bench_generator_args_match():
    """bench.make_scene must build what this file tests: compare the literal generator calls."""
    import inspect, bench
    src = inspect.getsource(bench.make_scene)
    for frag in ["n_instances=490, tree_subdiv=5", "max_bounces=16, subdiv=6, env=\"room_env.hdr\"",
                 "n_curves=10000, nodes_per_curve=67", "width=0.004", "cornell_dragon_standin(d, res=(W, H), spp=spp)",
                 "sky_envmap(512, 256)", "extent=40.0"]:
        assert frag in src, "bench.make_scene changed (%s): update tests/test_gpu_bench_scenes.py" % frag


# per-scene bars: (min fraction of pixels within 1e-5*(1+L) of the oracle, max RMSE / mean radiance, expected triangles,
# expected curve segments).  Measured values are in the comment; the bar is <= 3x the measured miss rate / RMSE.
BARS = {
    "c1": (0.9994, 4e-4, 868480, 0),     # measured (r02-a, B200): 0.99982 within tol, RMSE/mean 1.2e-4
    "c2": (0.9910, 2e-2, 327688, 0),     # measured: 0.99700, 6.6e-3 (4 x 81,920 furniture triangles + the 8-triangle mesh light)
    "c3": (0.9995, 1e-5, 12544000, 0),   # measured: 1.00000, 1.5e-7
    "c4": (0.970, 3e-2, 0, 650000),
}


@pytest.fixture(scope="module")
def scenes(tmp_path_factory):
    cache = {}

    def get(config, oracle=False):
        if config not in cache:
            d = str(tmp_path_factory.mktemp("bench_" + config))
            cache[config] = [scene.load_scene(_build(config, d)), None]
        if oracle:
            if cache[config][1] is None:
                cache[config][1] = pyoracle.Oracle(cache[config][0])     # (C3: the oracle's BVH build over 12.5 M triangles takes a while)
            return cache[config][1]
        return cache[config][0]
    yield get
    for fs, o in cache.values():
        if o is not None:
            o.close()


def test_generator_arguments_are_the_bench_ones():
    _bench_generator_args_match()


@pytest.mark.parametrize("config", ["c1", "c2", "c3", "c4"])
def test_bench_scene_matches_oracle(scenes, config):
    fs = scenes(config)
    frac_ok, rel_rmse, n_tris, n_segs = BARS[config]
    spp = 4
    ctx = lib.Context(fs)
    info = ctx.scene_info()
    assert info["n_tris"] == n_tris
    if n_segs:
        assert sum(p.n_curve_segments for p in fs.primitives if p.type == abi.PRIM_CURVES) == n_segs
    img, cnt = ctx.render_tiles(spp)
    st = ctx.stats()
    ctx.close()
    o = scenes(config, oracle=True)
    ref, rcnt = o.render(spp)
    d = np.abs(img - ref).max(axis=2)
    tol = 1e-5*(1.0 + np.abs(ref).max(axis=2))
    frac = float((d <= tol).mean()); exact = float((d == 0).mean())
    rmse = float(np.sqrt(((img - ref)**2).mean())); mean = float(ref.mean())
    print("%s: %d tris %d nodes depth %d | within tol %.5f exact %.5f rmse/mean %.3e | rays %d vs oracle %d" % (
        config, info["n_tris"], info["n_nodes"], info["bvh_depth"], frac, exact, rmse/max(mean, 1e-6), st.rays, o.stats.rays))
    assert np.array_equal(cnt, rcnt)
    assert np.isfinite(img).all() and mean > 1e-3
    assert frac >= frac_ok
    assert rmse <= rel_rmse*mean


@pytest.mark.parametrize("config", ["c1", "c3", "c4"])
def test_bench_scene_hit_ids(scenes, config):
    """200 k random rays through tgb200_trace_closest on the bench BVHs: primitive and triangle / segment ids equal to
    the oracle's (which walks its own median-split BVH2), exact-t ties excepted; t and backside bit-equal."""
    fs = scenes(config)
    rng = np.random.RandomState(11)
    n = 200000
    lo, hi = {"c1": ((-1.0, 0.0, -1.0), (1.0, 2.0, 1.0)), "c3": ((-40.0, 0.2, -40.0), (40.0, 8.0, 40.0)),
              "c4": ((-1.5, 0.2, -1.5), (1.5, 2.4, 1.5))}[config]
    o = np.stack([rng.uniform(lo[k], hi[k], n) for k in range(3)], axis=1).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32); d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = np.concatenate([o, d.astype(np.float32), np.full((n, 1), 5e-4, np.float32), np.full((n, 1), np.inf, np.float32)], axis=1)
    ref = scenes(config, oracle=True).trace(rays)
    ctx = lib.Context(fs); got = ctx.trace_closest(rays); ctx.close()
    same = (ref["primitive"] == got["primitive"]) & (ref["prim_id"] == got["prim_id"])
    with np.errstate(invalid="ignore"):
        tie = np.abs(ref["t"] - got["t"]) <= 4*np.spacing(np.abs(ref["t"]).astype(np.float32))
    hit = ref["primitive"] >= 0
    bad = ~same & ~tie
    print("%s: %d of %d rays hit; ids equal %.6f, ties %d, bad %d" % (config, hit.sum(), n, same.mean(), int((~same & tie).sum()), int(bad.sum())))
    assert hit.sum() > n//10
    if config == "c4":
        # curve hits depend on the farT a segment is entered with (reference's non-conservative bisection bound): >= 99.9 %
        assert same.mean() >= 0.999
    else:
        assert bad.sum() == 0
    assert np.array_equal(ref["t"][same], got["t"][same])
    assert np.array_equal(ref["backside"][same], got["backside"][same])


# ---- tile sharding on ONE device: pack -> concatenate -> unpack == unsharded render ------------------------------------
@pytest.mark.parametrize("world", [2, 8])
def test_shard_pack_gather_unpack_equals_unsharded(scenes, world):
    """The N-GPU data path of bench.py / tgb200_render_sharded, with the N ranks played one after the other by one
    device: every rank renders its tile share, tgb200_pack_tiles writes its send buffer, the buffers are concatenated the
    way ncclAllGather lays them out (rank-major, padded to the largest share), tgb200_unpack_tiles de-tiles every share
    into one framebuffer -> bit-identical to the one-rank render of the same samples."""
    import torch
    fs = scenes("c1")
    w, h = fs.resolution
    spp = 2
    ctx = lib.Context(fs)
    full, full_cnt = ctx.render_tiles(spp)
    tiles = integrator.dice_tiles(w, h, 0xBA5EBA11)
    for deal in ("round_robin", "morton"):
        shares = [integrator.shard_tiles(tiles, r, world, deal=deal) for r in range(world)]
        assert sorted((t.x, t.y) for s in shares for t in s) == sorted((t.x, t.y) for t in tiles)
        npix = [sum(t.w*t.h for t in s) for s in shares]
        slot = max(npix)*3
        gathered = torch.zeros(world*slot, dtype=torch.float32, device="cuda")
        for r in range(world):
            ctx.clear()
            ctx.render_resident(spp, tiles=shares[r])
            ctx.pack_tiles(shares[r], gathered.data_ptr() + 4*r*slot)
        torch.cuda.synchronize()
        ctx.clear()
        for r in range(world):
            ctx.unpack_tiles(shares[r], gathered.data_ptr() + 4*r*slot, spp)
        got, got_cnt = ctx.read_framebuffer()
        assert np.array_equal(got, full), deal
        assert np.array_equal(got_cnt, full_cnt), deal
    ctx.close()


def test_multi_device_context_equals_single_device(scenes):
    """tgb_settings::devices: the scene replicated on two GPUs of this process, tiles dealt in Morton order, shares gathered
    on devices[0] with peer copies -> the same framebuffer as one GPU, bit for bit; also through the host-buffer call and
    for an adaptive step (block records merged from the GPU that owns each tile)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    fs = scenes("c1")
    one = lib.Context(fs, device=0)
    a, ca = one.render_tiles(4)
    n_blocks = ((fs.resolution[0] + 3)//4)*((fs.resolution[1] + 3)//4)
    rec1 = (abi.SampleRecord*n_blocks)()
    for i, r in enumerate(rec1):
        r.next_sample_count = 1 + (i % 3); r.sample_index = 4
    one.render_adaptive(rec1)
    a2, ca2 = one.read_framebuffer()
    one.close()
    two = lib.Context(fs, devices=[0, 1])
    b, cb = two.render_tiles(4)
    assert np.array_equal(a, b) and np.array_equal(ca, cb)
    rec2 = (abi.SampleRecord*n_blocks)()
    for i, r in enumerate(rec2):
        r.next_sample_count = 1 + (i % 3); r.sample_index = 4
    two.render_adaptive(rec2)
    b2, cb2 = two.read_framebuffer()
    assert np.array_equal(a2, b2) and np.array_equal(ca2, cb2)
    assert bytes(rec1) == bytes(rec2)
    st = two.stats()
    assert st.samples >= fs.resolution[0]*fs.resolution[1]*4
    two.clear(); two.render_resident(2); c, _ = two.read_framebuffer()
    two.close()
    one = lib.Context(fs, device=0); one.render_resident(2); d, _ = one.read_framebuffer(); one.close()
    assert np.array_equal(c, d)
