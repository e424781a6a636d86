"""Host-side mirror of Fast4DMatrix::Vec3 (reference ext/fast_4d_matrix/fast_4d_matrix.c:29-305,
lib/fast_4d_matrix/fast_4d_matrix.rb:3-28).

This is the HOST representation of config vectors only (what ConfigurableObject produces and what
World/Camera hand to the C ABI).  The per-ray vector arithmetic of the hot path lives in the CUDA
kernels (raytracing_rb_b200/csrc), not here.  Quirks kept: `r2` is r*r (c:280-284), `cos` is |cos|
clamped to 1 and raises on a zero vector (c:109-129), `*`//`/` accept only Float scalars
(c:194,213), `to_s` prints 6 decimals (rb:7-13)."""
import math

from . import _edits


class Vec3:
    __slots__ = ("values", "_r")

    def __init__(self, x, y, z):
        self.values = [x, y, z]
        self._r = math.sqrt(x * x + y * y + z * z)

    @classmethod
    def from_a(cls, a, b, c):
        for v in (a, b, c):
            if not isinstance(v, float):
                raise TypeError("Vec3.from_a expects Floats (RFLOAT_VALUE, fast_4d_matrix.c:78-80)")
        return cls(a, b, c)

    def to_a(self):
        return list(self.values)

    def to_s(self, n=6):
        if n:
            return "[" + ", ".join(("%0." + str(n) + "f") % x for x in self.values) + "]"
        return str(self.values)

    __str__ = to_s

    def __repr__(self):
        return "Vec3" + self.to_s()

    def to_json(self, *_):
        import json
        return json.dumps(self.values)

    @property
    def r(self):
        return self._r

    @property
    def r2(self):
        return self._r * self._r

    def dot(self, o):
        a, b = self.values, o.values
        ret = 0.0
        ret += a[0] * b[0]
        ret += a[1] * b[1]
        ret += a[2] * b[2]
        return ret

    def cos(self, o):
        a, b = self.values, o.values
        ret = self.dot(o)
        r1 = a[0] * a[0] + a[1] * a[1] + a[2] * a[2]
        r2 = b[0] * b[0] + b[1] * b[1] + b[2] * b[2]
        if r1 == 0 or r2 == 0:
            raise RuntimeError("zero vector detected!")
        v = math.sqrt(ret * ret / r1 / r2)
        return 1.0 if v > 1 else v

    def cross(self, o):
        a, b = self.values, o.values
        return Vec3(a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0])

    def add(self, o):
        a, b = self.values, o.values
        return Vec3(a[0] + b[0], a[1] + b[1], a[2] + b[2])

    def sub(self, o):
        a, b = self.values, o.values
        return Vec3(a[0] - b[0], a[1] - b[1], a[2] - b[2])

    def mul(self, o):
        a = self.values
        if isinstance(o, float):
            return Vec3(a[0] * o, a[1] * o, a[2] * o)
        if not isinstance(o, Vec3):
            raise TypeError("wrong argument type %s (expected Vec3 or Float)" % type(o).__name__)
        b = o.values
        return Vec3(a[0] * b[0], a[1] * b[1], a[2] * b[2])

    def div(self, o):
        if not isinstance(o, float):
            raise ValueError("parameter must be float")  # rb_eArgError, c:220
        a = self.values
        return Vec3(a[0] / o, a[1] / o, a[2] / o)

    __add__, __sub__, __mul__, __truediv__ = add, sub, mul, div

    def __pos__(self):
        return Vec3(*self.values)

    def __neg__(self):
        a = self.values
        return Vec3(-a[0], -a[1], -a[2])

    def _recalc(self):  # after an in-place operation: a Vec3 of a world object or light may have changed
        _edits.touch()
        a = self.values
        self._r = math.sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2])
        return self

    def add_bang(self, o):  # add!
        for i in range(3):
            self.values[i] += o.values[i]
        return self._recalc()

    def sub_bang(self, o):  # sub!
        for i in range(3):
            self.values[i] -= o.values[i]
        return self._recalc()

    def mul_bang(self, o):  # mul!
        for i in range(3):
            self.values[i] *= (o if isinstance(o, float) else o.values[i])
        return self._recalc()

    def normalize(self):
        a = self.values
        r = math.sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2])
        if r == 0:
            raise RuntimeError("zero vector detected")
        return Vec3(a[0] / r, a[1] / r, a[2] / r)

    def normalize_bang(self):  # normalize!
        n = self.normalize()
        _edits.touch()
        self.values = n.values
        self._r = 1.0
        return self

    def __eq__(self, o):
        return isinstance(o, Vec3) and self.values == o.values

    def __iter__(self):
        return iter(self.values)
