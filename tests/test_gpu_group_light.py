"""Light propagation on a device group (aicb_group_light_*): the relaxation sharded by slabs of queue tiles.

The group keeps the single-scene contract (tests/test_gpu_light.py) against the oracle, and every member's replica is
byte-identical to every other's after every call.  Groups that name device 0 several times run the cross-slab
exchanges on one GPU; groups over distinct devices run when that many devices exist."""
import ctypes
import functools

import numpy as np
import pytest

import aicb200
import orc
from aicb200 import Block, DeviceGroup, GraphicsOptions, Space, SpaceRaytracer, abi, scenes
from test_gpu_light import NO_RAYS, OPAQUE, VISIBLE, WHITE, all_cubes, compare_fields, empty_space, light_scene

pytestmark = pytest.mark.gpu


def device_count():
    try:
        lib = ctypes.CDLL("libcuda.so.1")
        n = ctypes.c_int(0)
        if lib.cuInit(0) != 0 or lib.cuDeviceGetCount(ctypes.byref(n)) != 0:
            return 0
        return n.value
    except OSError:
        return 0


def _members():
    out = [pytest.param([0], id="0"), pytest.param([0, 0], id="0x2"), pytest.param([0, 0, 0], id="0x3"),
           pytest.param([0] * 5, id="0x5")]
    for n in (2, 4, 8):
        out.append(pytest.param(list(range(n)), id=f"devices{n}",
                                marks=pytest.mark.skipif(device_count() < n, reason=f"needs {n} devices")))
    return out


MEMBERS = _members()


def replicas(g):
    """Every member's light; asserts they are byte-identical and returns member 0's."""
    fields = [g.light_download(m) for m in range(g.size)]
    for m in range(1, g.size):
        assert np.array_equal(fields[m], fields[0]), f"member {m}'s replica differs from member 0's"
    return fields[0]


def check_stats(g, updates):
    total = g.light_stats()
    members = [g.light_stats(m) for m in range(g.size)]
    assert total["cube_updates"] == updates == sum(s["cube_updates"] for s in members)
    assert total["chart_node_visits"] == sum(s["chart_node_visits"] for s in members)
    assert all(s["rounds"] == total["rounds"] for s in members)


def group_of(members, space):
    g = DeviceGroup(members)
    g.update(space)
    return g


def flood_space():
    """tests/test_gpu_light.py::test_light_bench_shape_flood's 32^3 slice of C4 (32 queue tiles)."""
    n = 32
    h = scenes.grid_hash(21, (n, n, n))
    blocks = [Block.air()] + [Block(color=(0.3 + 0.1 * i, 0.8 - 0.1 * i, 0.5, 1.0)) for i in range(4)] + \
             [Block(color=(0.1, 0.1, 0.1, 1.0), emission=(3.0, 3.0, 2.0))]
    ids = np.where((h & np.uint64(15)) == 0, 1 + ((h >> np.uint64(8)) % np.uint64(5)).astype(np.int64), 0).astype(np.uint16)
    ids[:, : n // 4, :] = 1
    light = np.zeros((n, n, n, 4), dtype=np.uint8)
    light[..., 3] = NO_RAYS
    return Space((0, 0, 0), ids, blocks, light=light, sky_colors=scenes.OCTANT_SKY, light_max_distance=30)


def scene_edits(space, n, seed):
    rng = np.random.default_rng(seed)
    cubes = np.stack([rng.integers(0, space.size[a], n) + space.lower[a] for a in range(3)], axis=1).astype(np.int32)
    return cubes, rng.integers(0, len(space.blocks), n).astype(np.uint16)


SPACES = {"light_scene": light_scene, "light_scene_9": lambda: light_scene(seed=9), "flood": flood_space}
EDITS = {"light_scene": lambda sp: scene_edits(sp, 60, 4), "light_scene_9": lambda sp: scene_edits(sp, 60, 4),
         "flood": lambda sp: scene_edits(sp, 300, 1)}


@functools.lru_cache(maxsize=None)
def oracle_fields(name):
    """The oracle's converged field and its field after EDITS[name] (the same for every group: computed once)."""
    space = SPACES[name]()
    ol = orc.OracleLight(space)
    ol.fast_evaluate()
    ol.evaluate(0)
    converged = ol.field()
    ol.set_cubes(*EDITS[name](space))
    ol.evaluate(0)
    return converged, ol.field()


def converge_group(members, name):
    space = SPACES[name]()
    g = group_of(members, space)
    g.light_fast_evaluate()
    replicas(g)
    n, md, nv = g.light_evaluate(0)
    check_stats(g, n)
    return space, g


@pytest.mark.parametrize("members", MEMBERS)
def test_reference_light_kats_on_group(members):
    """light/tests.rs:233-261 exact neighbour values around an opaque emitter; `evaluate_light` counts 0 / 2 / 0."""
    light = (0.5, 1.0, 2.0)
    g = group_of(members, empty_space((3, 3, 3), [Block(color=WHITE, emission=light)], sky=[(0.0, 0.0, 0.0)]))
    g.light_edit_and_propagate([(1, 1, 1)], [1], 0)
    f = replicas(g)
    L = orc.lib()
    val = lambda t: tuple(np.float32(L.orc_packed_light_lut(int(v))) for v in t[:3])
    f32 = np.float32
    assert val(f[0, 1, 1]) == val(f[2, 1, 1]) == (f32(0.13397168), f32(0.26794338), f32(0.53588676))
    assert val(f[1, 0, 1]) == val(f[1, 2, 1]) == (f32(0.1649385), f32(0.32987696), f32(0.6597539))
    assert val(f[1, 1, 0]) == val(f[1, 1, 2]) == (f32(0.21763763), f32(0.43527526), f32(0.8705506))
    g = group_of(members, empty_space((3, 1, 1), [Block(color=WHITE)]))
    assert g.light_evaluate(0)[0] == 0
    assert g.light_edit_and_propagate([(1, 0, 0)], [1], 0)[0] == 2
    check_stats(g, 2)
    assert g.light_evaluate(0)[0] == 0
    replicas(g)
    g = group_of(members, empty_space((3, 1, 1), [Block(color=WHITE)], sky=[(1.0, 0.0, 0.0)]))
    n, md = g.light_edit_and_propagate([(0, 0, 0)], [1], 0)
    f = replicas(g)
    assert n == 1 and tuple(f[0, 0, 0]) == (0, 0, 0, OPAQUE) and tuple(f[2, 0, 0]) == (0, 0, 0, NO_RAYS)
    assert tuple(f[1, 0, 0]) == (144, 0, 0, VISIBLE)


@pytest.mark.parametrize("members", MEMBERS)
def test_converged_field_matches_oracle_and_is_quiescent(members):
    """14^3 = 3 queue tiles with max_distance 12: every slab is thinner than a cube's reach."""
    space, g = converge_group(members, "light_scene")
    gpu = replicas(g)
    compare_fields(gpu, oracle_fields("light_scene")[0])
    sp2 = Space(space.lower, space.block_ids, space.blocks, light=gpu, sky_colors=space.sky_colors, light_max_distance=12)
    again = SpaceRaytracer(sp2, GraphicsOptions()).light_compute(all_cubes(space)).reshape(gpu.shape)
    vis = gpu[..., 3] == VISIBLE
    d = np.abs(again[..., :3].astype(int) - gpu[..., :3].astype(int)).max(axis=-1)[vis]
    assert np.array_equal(again[..., 3][vis], gpu[..., 3][vis])
    assert (d == 0).mean() > 0.8 and d.max() <= 12, (float((d == 0).mean()), int(d.max()))


@pytest.mark.parametrize("members", MEMBERS)
def test_edits_then_propagate_matches_oracle_and_renders(members):
    space, g = converge_group(members, "light_scene_9")
    cubes, ids = EDITS["light_scene_9"](space)
    n, md = g.light_edit_and_propagate(cubes, ids, 0)
    assert n > 0
    check_stats(g, n)
    field = replicas(g)
    compare_fields(field, oracle_fields("light_scene_9")[1])
    # the group renders the edited Space and its light: identical to a fresh snapshot of both
    ids2 = space.block_ids.copy()
    for c, i in zip(cubes, ids):
        ids2[tuple(c - np.array(space.lower))] = i
    fresh = Space(space.lower, ids2, space.blocks, light=field, sky_colors=space.sky_colors, light_max_distance=12)
    opts = GraphicsOptions()
    cam = scenes.standard_camera(space, opts, 64, 48)
    r = aicb200.RtRenderer(cam)
    r.update(fresh)
    assert np.array_equal(g.draw(cam, opts).data, r.draw().data)


@pytest.mark.parametrize("members", MEMBERS)
def test_flood_with_edits_matches_oracle(members):
    """32^3 C4-shaped flood (32 tiles), then 300 random edits."""
    space, g = converge_group(members, "flood")
    converged, edited = oracle_fields("flood")
    compare_fields(replicas(g), converged)
    n, md = g.light_edit_and_propagate(*EDITS["flood"](space), 0)
    check_stats(g, n)
    compare_fields(replicas(g), edited)


def test_upload_light_and_update_blocks_reach_every_replica():
    space = light_scene()
    g = group_of([0, 0, 0], space)
    field = np.random.default_rng(2).integers(0, 256, space.size + (4,)).astype(np.uint8)
    g.upload_light(field)
    assert np.array_equal(replicas(g), field)
    # block 1 (the floor) becomes a light source: the group's propagation equals a single scene's of the same edit
    emitter = Block(color=(0.8, 0.7, 0.6, 1.0), emission=(2.0, 1.0, 0.5))
    g.update_blocks([1], [emitter])
    rt = SpaceRaytracer(space, GraphicsOptions())
    rt.upload_light(field)
    rt.update_blocks([1], [emitter])
    for target in (g, rt):
        target.light_fast_evaluate()
        target.light_evaluate(0)
    compare_fields(replicas(g), rt.light_download())
    g.update_cubes([(0, 3, 5)], [2], light=[(1, 2, 3, VISIBLE)])
    assert tuple(replicas(g)[2, 2, 2]) == (1, 2, 3, VISIBLE)


def test_invalid_calls_change_no_replica():
    sp = empty_space((4, 4, 4), [Block(color=WHITE)])
    sp.light_max_distance = 0   # LightPhysics::None
    g = group_of([0, 0], sp)
    with pytest.raises(aicb200.AicbError) as e:
        g.light_evaluate(0)
    assert e.value.status == abi.ERR_INVALID
    with pytest.raises(aicb200.AicbError) as e:
        g.light_edit_and_propagate([(1, 1, 1)], [1], 0)
    assert e.value.status == abi.ERR_INVALID
    space, g = converge_group([0, 0, 0], "light_scene")
    before = replicas(g)
    for cubes, ids in (([(0, 3, 5), (100, 0, 0)], [1, 1]), ([(0, 3, 5)], [len(space.blocks)])):
        with pytest.raises(aicb200.AicbError) as e:
            g.light_edit_and_propagate(cubes, ids, 0)
        assert e.value.status == abi.ERR_INVALID
        assert np.array_equal(replicas(g), before)
    # the host mirrors did not change either: a valid edit afterwards still matches a single scene
    rt = SpaceRaytracer(Space(space.lower, space.block_ids, space.blocks, light=before, sky_colors=space.sky_colors,
                              light_max_distance=12), GraphicsOptions())
    with pytest.raises(aicb200.AicbError):
        g.light_download(3)
    g.light_edit_and_propagate([(0, 3, 5)], [1], 0)
    rt.light_edit_and_propagate([(0, 3, 5)], [1], 0)
    compare_fields(replicas(g), rt.light_download())
