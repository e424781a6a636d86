"""Host-side checks of rtrb_scene_update: exported and declared without an ABI bump, a NULL renderer is an argument
error, and a scene the library rejects is rejected before any device is needed, exactly as rtrb_renderer_create
rejects it."""
import ctypes as C
import os
import subprocess

import pytest

from raytracing_rb_b200 import _abi
from helpers_rtrb import load_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "raytracing_rb_b200", "csrc"), "-j4", "-s", "all"])
    from raytracing_rb_b200 import _lib
    return _lib.lib()


def test_scene_update_is_exported_abi_unchanged(L):
    from raytracing_rb_b200 import Renderer, _lib
    assert "rtrb_scene_update" in _lib.EXPORTS and hasattr(L, "rtrb_scene_update")
    assert callable(Renderer.update)
    assert L.rtrb_abi_version() == _abi.ABI_VERSION == 4
    with open(os.path.join(ROOT, "include", "rtrb_b200.h")) as f:
        assert "int rtrb_scene_update(rtrb_renderer* r, const rtrb_scene_desc* scene, void* stream);" in f.read()


def test_null_renderer_is_invalid(L):
    world, _ = load_scene(2, width=8, height=4)
    holder = world.to_scene_desc()
    assert L.rtrb_scene_update(None, C.byref(holder.desc), None) == _abi.RTRB_ERR_INVALID
    assert b"renderer is NULL" in L.rtrb_last_error()


def _break(holder, how):
    o = holder.desc.objects[3]
    if how == "sphere_without_refractive_rate":
        o.has_refraction = 0
    elif how == "unknown_type":
        o.type = 7
    elif how == "bad_texture_index":
        o.texture = 5
    else:
        holder.desc.n_lights = 1000


@pytest.mark.parametrize("how", ["sphere_without_refractive_rate", "unknown_type", "bad_texture_index", "too_many_lights"])
def test_invalid_scene_is_rejected_as_create_rejects_it(L, how):
    world, _ = load_scene(2, width=8, height=4)
    holder = world.to_scene_desc()
    _break(holder, how)
    out = C.c_void_p()
    want = L.rtrb_renderer_create(C.byref(holder.desc), 0, C.byref(out))
    want_msg = L.rtrb_last_error()
    assert want in (_abi.RTRB_ERR_INVALID, _abi.RTRB_ERR_UNSUPPORTED) and not out.value
    assert L.rtrb_scene_update(None, C.byref(holder.desc), None) == want
    assert L.rtrb_last_error() == want_msg


class _FakeRenderer:
    def __init__(self):
        self.updates = 0
        self.synced_to = None

    def update(self, scene):
        self.updates += 1


def test_unchanged_world_is_not_flattened_again():
    """Camera.renderer() / World.renderer() re-flatten and update only after an edit of the scene mirror: attribute
    assignment on objects, lights and the World, list changes of world_objects / lights, in-place Vec3 operations."""
    from raytracing_rb_b200 import Vec3, world as world_mod
    world, _ = load_scene(2, width=8, height=4)
    fake = _FakeRenderer()
    rs = {0: fake}
    calls = []
    real = world.to_scene_desc
    world.to_scene_desc = lambda: calls.append(1) or real()

    def sync():
        assert world_mod.synced_renderer(rs, 0, world) is fake
        return fake.updates

    assert sync() == 1          # never synced with this world
    assert sync() == 1 and sync() == 1
    assert len(calls) == 1      # unchanged: not flattened again
    edits = [lambda: setattr(world.world_objects[3], "radius", 0.5),
             lambda: setattr(world.lights[0], "color", Vec3(0.5, 0.5, 0.5)),
             lambda: world.world_objects[4].center.add_bang(Vec3(0.1, 0.0, 0.0)),
             lambda: world.world_objects.append(world.world_objects[1]),
             lambda: world.world_objects.pop(),
             lambda: world.lights.__setitem__(0, world.lights[0]),
             lambda: setattr(world, "max_distance", 500.0),
             lambda: setattr(world, "world_objects", list(world.world_objects))]
    for i, edit in enumerate(edits):
        edit()
        assert sync() == 2 + i, i
        assert sync() == 2 + i, i
    other, _ = load_scene(2, width=8, height=4)
    assert world_mod.synced_renderer(rs, 0, other) is fake and fake.updates == 2 + len(edits)  # another world
