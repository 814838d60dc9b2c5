"""Light propagation in budgeted steps (aicb_light_step) and the list of cubes whose light changed
(aicb_light_take_changes), on a scene and on a device group.

A step without a budget relaxes exactly as aicb_light_evaluate / aicb_light_edit_and_propagate; a budgeted step takes
at most its cap of cube updates and, when it took fewer, leaves nothing above epsilon queued; a drain of budgeted steps
keeps the oracle contract of tests/test_gpu_light.py.  The queue report is pinned on the oracle's queue."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import aicb200
import orc
from aicb200 import Block, GraphicsOptions, SpaceRaytracer, abi
from test_gpu_group_light import EDITS, MEMBERS, SPACES, group_of, oracle_fields, replicas
from test_gpu_light import NO_RAYS, VISIBLE, WHITE, compare_fields, empty_space, light_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS_PRIORITY = 1   # Priority::from_difference(0): a queue whose highest priority is <= 1 holds nothing above epsilon 0


def test_light_updates_layout_matches_c_header(tmp_path):
    src = tmp_path / "layout.c"
    fields = [f[0] for f in abi.LightUpdates._fields_]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "aicb200.h"\nint main(){printf("%zu'
                   + " %zu" * len(fields) + '\\n", sizeof(aicb_light_updates)'
                   + "".join(f", offsetof(aicb_light_updates, {f})" for f in fields) + ");return 0;}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [C.sizeof(abi.LightUpdates)] + [getattr(abi.LightUpdates, f).offset for f in fields]
    assert got[0] == 40


def scene(space):
    return SpaceRaytracer(space, GraphicsOptions())


def stats_of(target):
    st = target.light_stats()
    return st["cube_updates"], st["chart_node_visits"], st["rounds"]


def drain(target, cap, max_steps=200_000, check=None, **step_args):
    """Steps with max_updates=cap until nothing above epsilon is queued; every step keeps the cap contract."""
    infos = []
    info = target.light_step(max_updates=cap, **step_args)
    while True:
        infos.append(info)
        assert info["update_count"] <= cap, (info, cap)
        if info["update_count"] < cap:
            assert info["max_queue_priority"] <= EPS_PRIORITY, info
        if check:
            check(info)
        if info["max_queue_priority"] <= EPS_PRIORITY:
            return infos
        assert len(infos) < max_steps, "the drain does not end"
        info = target.light_step(max_updates=cap)


# ---- 1. a step without a budget is evaluate_light ----------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["light_scene", "light_scene_9", "flood"])
def test_unbudgeted_step_equals_evaluate(name):
    space = SPACES[name]()
    a, b, c = scene(space), scene(space), scene(space)
    for t in (a, b, c):
        t.light_fast_evaluate()
    a.light_evaluate(0)
    b.light_evaluate(0)
    # the control: the apply kernel's guesses are a CAS race, so first check that evaluate reproduces itself here
    assert np.array_equal(a.light_download(), b.light_download()), "two evaluate_light runs differ: no control"
    assert stats_of(a) == stats_of(b)
    info = c.light_step(epsilon=0)
    assert np.array_equal(c.light_download(), a.light_download())
    assert (info["update_count"], info["chart_node_visits"], info["rounds"]) == stats_of(a) == stats_of(c)
    assert info["max_queue_priority"] <= EPS_PRIORITY
    cubes, ids = EDITS[name](space)
    a.light_edit_and_propagate(cubes, ids, 0)
    b.light_edit_and_propagate(cubes, ids, 0)
    assert np.array_equal(a.light_download(), b.light_download()), "two edit_and_propagate runs differ: no control"
    info = c.light_step(cubes, ids, epsilon=0)
    assert np.array_equal(c.light_download(), a.light_download())
    assert (info["update_count"], info["chart_node_visits"], info["rounds"]) == stats_of(a) == stats_of(c)


# ---- 2. the queue report -------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_queue_report_matches_oracle():
    space = light_scene()
    ol = orc.OracleLight(space)
    ol.fast_evaluate()
    rt = scene(space)
    rt.light_fast_evaluate()
    before = rt.light_download()
    info = rt.light_step(max_updates=0)
    assert info["update_count"] == 0 and info["rounds"] == 0
    assert np.array_equal(rt.light_download(), before)
    assert info["queue_count"] == ol.queue_len() > 0
    assert info["max_queue_priority"] == ol.queue_peek()
    assert rt.light_stats()["cube_updates"] == 0
    cubes, ids = EDITS["light_scene"](space)
    ol.set_cubes(cubes, ids)
    info = rt.light_step(cubes, ids, max_updates=0)
    assert info["update_count"] == 0 and info["rounds"] == 0
    assert (info["queue_count"], info["max_queue_priority"]) == (ol.queue_len(), ol.queue_peek())
    # an invalid edit list changes neither the light nor the queue
    edited = rt.light_download()
    for bad_cubes, bad_ids in (([(0, 3, 5), (100, 0, 0)], [1, 1]), ([(0, 3, 5)], [len(space.blocks)])):
        with pytest.raises(aicb200.AicbError) as e:
            rt.light_step(bad_cubes, bad_ids)
        assert e.value.status == abi.ERR_INVALID
        assert np.array_equal(rt.light_download(), edited)
    info = rt.light_step(max_updates=0)
    assert (info["queue_count"], info["max_queue_priority"]) == (ol.queue_len(), ol.queue_peek())
    with pytest.raises(aicb200.AicbError) as e:
        rt.light_step(budget_us=float("nan"))
    assert e.value.status == abi.ERR_INVALID
    none = empty_space((4, 4, 4), [Block(color=WHITE)])
    none.light_max_distance = 0   # LightPhysics::None
    with pytest.raises(aicb200.AicbError) as e:
        scene(none).light_step()
    assert e.value.status == abi.ERR_INVALID


# ---- 3. budgets hold and converge ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,cap", [("light_scene", 1), ("light_scene", 7), ("light_scene", 64), ("light_scene", 1000),
                                      ("flood", 500), ("flood", 5000), ("flood", 100)])
def test_budgeted_drain_holds_its_caps_and_converges(name, cap):
    """flood: 100 is below the band count of a single tile early in the drain, so rounds stop inside a tile."""
    space = SPACES[name]()
    rt = scene(space)
    rt.light_fast_evaluate()
    infos = drain(rt, cap, epsilon=0)
    assert sum(i["update_count"] for i in infos) > 0
    assert rt.light_stats()["cube_updates"] == infos[-1]["update_count"]
    compare_fields(rt.light_download(), oracle_fields(name)[0])


# ---- 4. the reference's KATs under budgets -------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1, 2])
def test_reference_kats_under_budgets(cap):
    light = (0.5, 1.0, 2.0)
    rt = scene(empty_space((3, 3, 3), [Block(color=WHITE, emission=light)], sky=[(0.0, 0.0, 0.0)]))
    drain(rt, cap, cubes=[(1, 1, 1)], block_ids=[1])
    f = rt.light_download()
    L = orc.lib()
    val = lambda t: tuple(np.float32(L.orc_packed_light_lut(int(v))) for v in t[:3])
    f32 = np.float32
    assert val(f[0, 1, 1]) == val(f[2, 1, 1]) == (f32(0.13397168), f32(0.26794338), f32(0.53588676))
    assert val(f[1, 0, 1]) == val(f[1, 2, 1]) == (f32(0.1649385), f32(0.32987696), f32(0.6597539))
    assert val(f[1, 1, 0]) == val(f[1, 1, 2]) == (f32(0.21763763), f32(0.43527526), f32(0.8705506))


@pytest.mark.gpu
def test_three_cube_line_steps_one_update_at_a_time():
    rt = scene(empty_space((3, 1, 1), [Block(color=WHITE)]))
    info = rt.light_step([(1, 0, 0)], [1], max_updates=1)
    assert (info["update_count"], info["queue_count"]) == (1, 1)
    info = rt.light_step(max_updates=1)
    assert (info["update_count"], info["queue_count"], info["max_queue_priority"]) == (1, 0, 0)
    # budget_us = 0 relaxes nothing, like max_updates = 0
    rt = scene(empty_space((3, 1, 1), [Block(color=WHITE)]))
    info = rt.light_step([(1, 0, 0)], [1], budget_us=0)
    assert (info["update_count"], info["rounds"], info["queue_count"]) == (0, 0, 2)
    # a positive time budget drains to the same light as one unbudgeted propagation
    ref = scene(empty_space((3, 1, 1), [Block(color=WHITE)]))
    assert ref.light_edit_and_propagate([(1, 0, 0)], [1], 0)[0] == 2
    for _ in range(10):
        info = rt.light_step(budget_us=5.0)
        assert info["update_count"] >= 1 or info["max_queue_priority"] <= EPS_PRIORITY
        if info["max_queue_priority"] <= EPS_PRIORITY:
            break
    assert info["queue_count"] == 0
    assert np.array_equal(rt.light_download(), ref.light_download())


@pytest.mark.gpu
def test_time_budget_drains_to_the_oracle_contract():
    space = light_scene()
    rt = scene(space)
    rt.light_fast_evaluate()
    for _ in range(100_000):
        info = rt.light_step(budget_us=30.0)
        assert info["update_count"] >= 1 or info["max_queue_priority"] <= EPS_PRIORITY
        if info["max_queue_priority"] <= EPS_PRIORITY:
            break
    assert info["max_queue_priority"] <= EPS_PRIORITY
    compare_fields(rt.light_download(), oracle_fields("light_scene")[0])


# ---- 5. the change list --------------------------------------------------------------------------------------------
def host_diff(space, prev, cur):
    idx = np.argwhere((cur != prev).any(axis=-1))   # C order of [x, y, z] = increasing Z-major linear index
    return (idx + np.array(space.lower)).astype(np.int32), cur[tuple(idx.T)]


def check_take(target, space, prev, cur):
    cubes, texels = target.light_take_changes()
    want_cubes, want_texels = host_diff(space, prev, cur)
    assert np.array_equal(cubes, want_cubes)
    assert np.array_equal(texels, want_texels)
    empty = target.light_take_changes()
    assert empty[0].shape == (0, 3) and empty[1].shape == (0, 4), "a second take is not empty"
    return len(cubes)


@pytest.mark.gpu
def test_change_list_equals_the_host_diff():
    space = light_scene()
    assert space.lower != (0, 0, 0)
    rt = scene(space)
    with pytest.raises(aicb200.AicbError) as e:
        rt.light_take_changes()
    assert e.value.status == abi.ERR_INVALID
    rt.light_track_changes(True)
    prev = rt.light_download()
    rt.light_fast_evaluate()
    cur = rt.light_download()
    assert check_take(rt, space, prev, cur) > 0
    for _ in range(3):
        prev = cur
        rt.light_step(max_updates=500)
        cur = rt.light_download()
        assert check_take(rt, space, prev, cur) > 0
    # a cap that is too small consumes nothing
    prev = cur
    rt.light_step(*EDITS["light_scene"](space), max_updates=300)
    cur = rt.light_download()
    n = C.c_size_t(0)
    lib = aicb200.load_library()
    aicb200._check(lib.aicb_light_take_changes(rt.handle, None, None, 0, C.byref(n)))
    assert n.value > 1
    small_c, small_t = np.zeros((n.value - 1, 3), np.int32), np.zeros((n.value - 1, 4), np.uint8)
    m = C.c_size_t(0)
    aicb200._check(lib.aicb_light_take_changes(rt.handle, small_c.ctypes.data, small_t.ctypes.data, n.value - 1, C.byref(m)))
    assert m.value == n.value and not small_c.any() and not small_t.any()
    check_take(rt, space, prev, cur)
    # upload_light and update_cubes with light are changes too
    prev = cur
    field = cur.copy()
    field[3:7, 2:5, 1:9] = np.random.default_rng(5).integers(0, 256, (4, 3, 8, 4)).astype(np.uint8)
    rt.upload_light(field)
    cur = rt.light_download()
    assert check_take(rt, space, prev, cur) > 0
    prev = cur
    rt.update_cubes([(0, 3, 5), (3, 2, 4)], [2, 0], light=[(1, 2, 3, VISIBLE), (9, 8, 7, NO_RAYS)])
    cur = rt.light_download()
    assert check_take(rt, space, prev, cur) == 2
    # disabled: taking is invalid; re-enabling resets the baseline
    rt.light_track_changes(False)
    with pytest.raises(aicb200.AicbError) as e:
        rt.light_take_changes()
    assert e.value.status == abi.ERR_INVALID
    rt.upload_light(prev)
    rt.light_track_changes(True)
    assert len(rt.light_take_changes()[0]) == 0
    rt.light_step(max_updates=200)
    check_take(rt, space, prev, rt.light_download())


# ---- 6. groups -----------------------------------------------------------------------------------------------------
def check_group_counts(g, info):
    total = g.light_stats()
    members = [g.light_stats(m) for m in range(g.size)]
    assert info["update_count"] == total["cube_updates"] == sum(s["cube_updates"] for s in members)
    assert info["chart_node_visits"] == total["chart_node_visits"] == sum(s["chart_node_visits"] for s in members)
    assert info["rounds"] == total["rounds"]


@pytest.mark.gpu
@pytest.mark.parametrize("members", MEMBERS)
def test_group_steps(members):
    space = SPACES["light_scene"]()
    a, b, c = (group_of(members, space) for _ in range(3))
    for g in (a, b, c):
        g.light_fast_evaluate()
    ol = orc.OracleLight(space)
    ol.fast_evaluate()
    info = c.light_step(max_updates=0)
    assert (info["queue_count"], info["max_queue_priority"]) == (ol.queue_len(), ol.queue_peek())
    a.light_evaluate(0)
    b.light_evaluate(0)
    assert np.array_equal(replicas(a), replicas(b)), "two group evaluate_light runs differ: no control"
    c.light_track_changes(True)
    prev = replicas(c)
    info = c.light_step()
    check_group_counts(c, info)
    cur = replicas(c)
    assert np.array_equal(cur, replicas(a))
    assert info["update_count"] == a.light_stats()["cube_updates"] and info["rounds"] == a.light_stats()["rounds"]
    check_take(c, space, prev, cur)
    # budgeted drains: every replica identical after every step, counts summed over the members
    for name, cap in (("light_scene", 7), ("flood", 1000)):
        space = SPACES[name]()
        g = group_of(members, space)
        g.light_fast_evaluate()
        g.light_track_changes(True)
        prev = replicas(g)

        def check(info):
            nonlocal prev
            check_group_counts(g, info)
            cur = replicas(g)
            check_take(g, space, prev, cur)
            prev = cur
        drain(g, cap, check=check)
        compare_fields(replicas(g), oracle_fields(name)[0])
