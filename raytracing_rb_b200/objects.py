"""Mirror of Alex::Objects::{WorldObject,Sphere,Plane,Box} (reference src/objects/world_object.rb:8-18,
sphere.rb:6-26, plane.rb:7-36, box.rb:9-74) as HOST-side property bags: same attribute names, same derived
vectors, same mandatory-in-practice keys.  Their per-ray methods (intersect, cover_area,
local_lighting, ...) are the CUDA kernels' job; `to_desc` flattens one object for the C ABI."""
from . import _abi
from ._edits import Tracked
from .texture import Texture
from .vec3 import Vec3


def _f(x, what):
    if x is None:
        raise TypeError("%s is required (the reference would raise NoMethodError/TypeError on nil)" % what)
    return float(x)


def _v(x, what):
    if not isinstance(x, Vec3):
        raise TypeError("%s must be a 3-element numeric array" % what)
    return (_abi.D3)(*x.to_a())


class WorldObject(Tracked):
    # world_object.rb:9-13 accessors (nil when absent)
    name = None
    reflective_attenuation = refractive_attenuation = diffuse_rate = ambient = None
    refractive_rate = None
    texture_file_path = texture_horizontal_scale = texture_vertical_scale = None
    texture_u_offset = texture_v_offset = None
    texture = None
    TYPE = None

    def __init__(self, properties=None, config_path=None):  # world_object.rb:14-18
        self._config_path = config_path
        for key, value in (properties or {}).items():
            setattr(self, key, value)

    def _material_into(self, d):
        what = "%s(%s)" % (type(self).__name__, self.name)
        d.diffuse_rate = _v(self.diffuse_rate, what + ".diffuse_rate")
        d.reflective_attenuation = _v(self.reflective_attenuation, what + ".reflective_attenuation")  # ray_tracer.rb:99
        d.ambient = _v(self.ambient, what + ".ambient")
        if self.refractive_attenuation is not None:
            d.refractive_attenuation = _v(self.refractive_attenuation, what + ".refractive_attenuation")
        elif d.has_refraction:
            raise TypeError(what + ": refractive_rate given without refractive_attenuation (ray_tracer.rb:117 would raise)")


class Sphere(WorldObject):  # sphere.rb
    TYPE = _abi.OBJ_SPHERE
    center = radius = None
    north_pole_vec = greenwich_vec = None
    ninety_degree_east_vec = None

    def __init__(self, properties=None, config_path=None):
        super().__init__(properties, config_path)
        if self.texture_file_path:  # sphere.rb:18-21
            self.ninety_degree_east_vec = self.north_pole_vec.cross(self.greenwich_vec)
            self.init_texture(self.texture_file_path)

    def init_texture(self, file_path):  # sphere.rb:24-26
        self.texture = Texture(file_path, self.texture_horizontal_scale, self.texture_vertical_scale,
                               self.texture_u_offset, self.texture_v_offset, config_path=self._config_path)

    def to_desc(self, texture_index):
        d = _abi.ObjectDesc()
        what = "Sphere(%s)" % self.name
        d.type = self.TYPE
        d.texture = texture_index
        d.has_refraction = 1
        d.point = _v(self.center, what + ".center")
        d.radius = _f(self.radius, what + ".radius")
        d.refractive_rate = _f(self.refractive_rate, what + ".refractive_rate")  # sphere.rb:93 divides unconditionally
        if self.refractive_attenuation is None:
            raise TypeError(what + ".refractive_attenuation is required for spheres")
        if texture_index >= 0:
            d.greenwich_vec = _v(self.greenwich_vec, what + ".greenwich_vec")
            d.north_pole_vec = _v(self.north_pole_vec, what + ".north_pole_vec")
            d.texture_horizontal_scale = _f(self.texture_horizontal_scale, what + ".texture_horizontal_scale")
            d.texture_vertical_scale = _f(self.texture_vertical_scale, what + ".texture_vertical_scale")
            d.texture_u_offset = float(self.texture.u_off)
            d.texture_v_offset = float(self.texture.v_off)
        self._material_into(d)
        return d


class Plane(WorldObject):  # plane.rb
    TYPE = _abi.OBJ_PLANE
    point = front = up = None
    u_unit = v_unit = None
    left = None

    def __init__(self, properties=None, config_path=None):
        if properties is None:  # Plane.create_from_scratch, plane.rb:17-19,25-26
            super().__init__({}, config_path)
            return
        super().__init__(properties, config_path)
        if self.texture_file_path:
            self.init_texture(self.texture_file_path)
        self.reinit()

    @classmethod
    def create_from_scratch(cls):
        return cls()

    def reinit(self):  # plane.rb:21-23
        self.left = self.front.cross(self.up).normalize()

    def init_texture(self, file_path):  # plane.rb:34-36
        self.texture = Texture(file_path, self.texture_horizontal_scale, self.texture_vertical_scale,
                               config_path=self._config_path)

    def to_desc(self, texture_index):
        d = _abi.ObjectDesc()
        what = "Plane(%s)" % self.name
        d.type = self.TYPE
        d.texture = texture_index
        d.has_refraction = 1 if self.refractive_rate is not None else 0  # plane.rb:57 `if self.refractive_rate` (0.0 is truthy in Ruby)
        d.point = _v(self.point, what + ".point")
        d.front = _v(self.front, what + ".front")
        d.up = _v(self.up, what + ".up")
        if texture_index >= 0:
            d.u_unit = _f(self.u_unit, what + ".u_unit")
            d.v_unit = _f(self.v_unit, what + ".v_unit")
            d.texture_horizontal_scale = _f(self.texture_horizontal_scale, what + ".texture_horizontal_scale")
            d.texture_vertical_scale = _f(self.texture_vertical_scale, what + ".texture_vertical_scale")
        else:
            d.u_unit = float(self.u_unit) if self.u_unit is not None else 1.0
            d.v_unit = float(self.v_unit) if self.v_unit is not None else 1.0
        if d.has_refraction:
            d.refractive_rate = float(self.refractive_rate)
        self._material_into(d)
        return d


class Box(WorldObject):  # box.rb
    """Six bounded faces (box.rb:22-73).  The faces are Plane.create_from_scratch objects carrying only
    what Box#initialize assigns; they are rebuilt here for introspection (`planes`), while the device
    derives its own copy from the same nine numbers in the reference's evaluation order."""
    TYPE = _abi.OBJ_BOX
    point = front = up = None
    width_front = width_up = width_left = None

    def __init__(self, properties=None, config_path=None):
        super().__init__(properties, config_path)
        if self.texture_file_path:  # box.rb:17-19: decoded, but Box never samples it (no local_lighting override)
            self.texture = Texture(self.texture_file_path, self.texture_horizontal_scale, self.texture_vertical_scale,
                                   config_path=self._config_path)
        left = self.front.cross(self.up).normalize()  # box.rb:23 (raises on a zero vector like the reference)
        wf, wu, wl = float(self.width_front), float(self.width_up), float(self.width_left)
        spec = [  # (front, up, point, u_unit, v_unit), box.rb:25-59
            (self.up, left, self.point + self.up * wu * 0.5, wf, wl),
            (-self.up, left, self.point - self.up * wu * 0.5, wf, wl),
            (self.front, self.up, self.point + self.front * wf * 0.5, wl, wu),
            (-self.front, self.up, self.point - self.front * wf * 0.5, wl, wu),
            (left, self.up, self.point + left * wl * 0.5, wf, wu),
            (-left, self.up, self.point - left * wl * 0.5, wf, wu),
        ]
        self.planes = []
        for f, u, pt, uu, vu in spec:
            p = Plane.create_from_scratch()
            p.front, p.up, p.point, p.u_unit, p.v_unit = f, u, pt, uu, vu
            p.reflective_attenuation = self.reflective_attenuation  # box.rb:66-72
            p.refractive_attenuation = self.refractive_attenuation
            p.refractive_rate = self.refractive_rate
            p.diffuse_rate = self.diffuse_rate
            p.reinit()
            self.planes.append(p)

    def to_desc(self, texture_index):
        d = _abi.ObjectDesc()
        what = "Box(%s)" % self.name
        d.type = self.TYPE
        d.texture = -1  # WorldObject#local_lighting runs without a colour filter for boxes
        d.has_refraction = 1 if self.refractive_rate is not None else 0  # plane.rb:57 on every face
        d.point = _v(self.point, what + ".point")
        d.front = _v(self.front, what + ".front")
        d.up = _v(self.up, what + ".up")
        d.width_front = _f(self.width_front, what + ".width_front")
        d.width_up = _f(self.width_up, what + ".width_up")
        d.width_left = _f(self.width_left, what + ".width_left")
        if d.has_refraction:
            d.refractive_rate = float(self.refractive_rate)
        self._material_into(d)
        return d


OBJECT_CLASSES = {"Sphere": Sphere, "Plane": Plane, "Box": Box}  # world.rb:31 `eval("Alex::Objects::#{type}")`
