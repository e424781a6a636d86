"""Mirror of Alex::World (reference src/world.rb:10-34): YAML -> objects + lights.  The scene
queries World#intersect / lit_area / local_lights / high_lights (:37-98) are device code; this
class builds the flat scene description handed to rtrb_renderer_create, and World#intersect is reachable on its own
through `intersect` / `intersect_batch` (rtrb_intersect_rays)."""
import ctypes as C

from .vec3 import Vec3

from . import _abi, _edits
from .configurable_object import ConfigurableObject
from .lights import LIGHT_CLASSES
from .objects import OBJECT_CLASSES


class SceneDescHolder:
    """A SceneDesc plus the Python objects that own the memory it points to."""

    def __init__(self, desc, keepalive):
        self.desc = desc
        self._keepalive = keepalive


def synced_renderer(renderers, device, world):
    """renderers[device]: made from `world` on first use, and brought up to date (rtrb_scene_update) when the world
    is another one or the scene mirror was edited since (_edits).  An unchanged world costs an integer compare."""
    stamp = _edits.count()  # before flattening: an edit made meanwhile is picked up by the next call
    r = renderers.get(device)
    if r is None:
        from .renderer import Renderer
        renderers[device] = r = Renderer(world.to_scene_desc(), device)
    elif r.synced_to != (world, stamp):
        r.update(world.to_scene_desc())
    r.synced_to = (world, stamp)
    return r


class World(ConfigurableObject):
    max_distance = None
    trace_depth = None          # world.rb:12, unused upstream (depth comes from the camera)
    soft_shadow_exponent = None

    def __init__(self, config_file):
        super().__init__(config_file)
        self.world_objects = self.parse_objects(self.world_objects)  # world.rb:17
        self.lights = self.parse_lights(self.lights)                  # world.rb:18

    def __setattr__(self, name, value):
        if name in ("world_objects", "lights") and isinstance(value, list) and not isinstance(value, _edits.TrackedList):
            value = _edits.TrackedList(value)
        _edits.touch()
        object.__setattr__(self, name, value)

    def renderer(self, device=0):
        """The scene baked on `device` for ray-level queries (one per device, made on first use), brought up to date
        with edits of the objects and lights since the last call."""
        return synced_renderer(self.__dict__.setdefault("_renderers", {}), device, self)

    def intersect_batch(self, rays, precision=_abi.PREC_DEFAULT, device=0):
        """World#intersect on many rays (Ray objects or [n, 6] rows of position, front) -> RAY_HIT_DTYPE array."""
        from .ray_tracer import rays_array
        return self.renderer(device).intersect_rays(rays_array(rays), precision)

    def intersect(self, ray, precision=_abi.PREC_DEFAULT, device=0):
        """world.rb:37-59 -> (object, intersection, direction, delta) as the reference returns them: the winning world
        object, Vec3, "in" / "out", Vec3; four Nones on a miss."""
        h = self.intersect_batch([ray], precision, device)[0]
        if h["object"] < 0:
            return None, None, None, None
        return (self.world_objects[int(h["object"])], Vec3(*[float(v) for v in h["intersection"]]),
                "in" if h["direction"] else "out", Vec3(*[float(v) for v in h["delta"]]))

    def parse_lights(self, array):  # world.rb:21-27
        ret = []
        for item in array:
            klass = LIGHT_CLASSES.get(str(item["type"]))
            if klass is None:
                raise NameError("uninitialized constant Alex::Lights::%sLight" % item["type"])
            ret.append(klass(item["properties"]))
        return ret

    def parse_objects(self, array):  # world.rb:28-34
        ret = []
        for item in array:
            klass = OBJECT_CLASSES.get(str(item["type"]))
            if klass is None:
                raise NameError("uninitialized constant Alex::Objects::%s" % item["type"])
            ret.append(klass(item["properties"], config_path=self.config_path))
        return ret

    def to_scene_desc(self):
        textures, tex_index, keep = [], {}, []
        objs = (_abi.ObjectDesc * max(1, len(self.world_objects)))()
        for i, o in enumerate(self.world_objects):
            ti = -1
            if o.texture is not None and getattr(o, "TYPE", None) != _abi.OBJ_BOX:
                key = o.texture.file_name
                if key not in tex_index:
                    tex_index[key] = len(textures)
                    textures.append(o.texture)
                ti = tex_index[key]
            objs[i] = o.to_desc(ti)
        lights = (_abi.LightDesc * max(1, len(self.lights)))()
        for i, l in enumerate(self.lights):
            d = _abi.LightDesc()
            d.position = (_abi.D3)(*l.position.to_a())
            d.color = (_abi.D3)(*l.color.to_a())
            d.radius = float(l.radius)
            d.high_light_rate = float(l.high_light_rate)
            d.high_light_angle = float(l.high_light_angle)
            lights[i] = d
        texs = (_abi.TextureDesc * max(1, len(textures)))()
        for i, t in enumerate(textures):
            texs[i].width, texs[i].height = t.width, t.height
            texs[i].rgb8 = t.rgb8.ctypes.data_as(C.POINTER(C.c_uint8))
            keep.append(t.rgb8)
        sd = _abi.SceneDesc()
        sd.max_distance = float(self.max_distance)
        sd.soft_shadow_exponent = float(self.soft_shadow_exponent)
        sd.n_objects, sd.n_lights, sd.n_textures = len(self.world_objects), len(self.lights), len(textures)
        sd.objects = C.cast(objs, C.POINTER(_abi.ObjectDesc))
        sd.lights = C.cast(lights, C.POINTER(_abi.LightDesc))
        sd.textures = C.cast(texs, C.POINTER(_abi.TextureDesc))
        keep += [objs, lights, texs, textures]
        return SceneDescHolder(sd, keep)
