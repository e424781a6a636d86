"""Edit counter of the scene mirror.  Camera.renderer() and World.renderer() re-flatten a world and hand it to
rtrb_scene_update only when the counter moved since their renderer was last brought up to date, so an unchanged world
costs one integer compare per call instead of World.to_scene_desc() (milliseconds for a thousand objects).

The counter moves on every attribute assignment of a world object, light, texture or World, on every change of the
World's world_objects / lights lists, and on the in-place Vec3 operations (add!, sub!, mul!, normalize!).  Writes that
bypass these (numpy edits of Texture.rgb8, item assignment into Vec3.values) are not seen: call touch() after them."""

_count = 0


def count():
    return _count


def touch():
    """Marks the scene mirror as edited."""
    global _count
    _count += 1


class Tracked:
    """Base of the mirror classes whose attributes make up the baked scene."""

    def __setattr__(self, name, value):
        touch()
        object.__setattr__(self, name, value)


class TrackedList(list):
    """A list whose in-place changes count as scene edits (World.world_objects / World.lights)."""


def _tracking(name):
    method = getattr(list, name)

    def wrapped(self, *args, **kw):
        touch()
        return method(self, *args, **kw)
    wrapped.__name__ = name
    return wrapped


for _name in ("__setitem__", "__delitem__", "__iadd__", "__imul__", "append", "extend", "insert", "pop", "remove",
              "clear", "sort", "reverse"):
    setattr(TrackedList, _name, _tracking(_name))
