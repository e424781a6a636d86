"""Mirror of Alex::Texture (reference src/objects/texture.rb:8-28), host side only: decode once
(PIL instead of RMagick) into 8-bit RGB rows.  The reference stores `(q16 >> 8) / 256.0` (:19),
which for an 8-bit source is v8/256.0; the device keeps the bytes and divides on lookup.  The
nearest-texel lookup `color(u, v)` runs on the device; `texel_index` restates its index rule for
host-side tooling."""
import math
import os

import numpy as np

from ._edits import Tracked


def resolve_texture_path(file_name, config_path=None):
    """The reference opens the path relative to the process CWD (texture.rb:12).  Fall back to the
    config file's project root and to this repository's root so shipped configs keep working."""
    cands = [file_name]
    if config_path:
        base = os.path.dirname(os.path.abspath(config_path))
        cands += [os.path.join(base, file_name), os.path.join(os.path.dirname(base), file_name)]
    cands.append(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), file_name))
    for c in cands:
        if os.path.isfile(c):
            return c
    raise FileNotFoundError("texture file not found: %s (tried %s)" % (file_name, cands))


class Texture(Tracked):
    def __init__(self, file_name, horizontal_scale, vertical_scale, u_off=None, v_off=None, config_path=None):
        from PIL import Image
        self.file_name = resolve_texture_path(file_name, config_path)
        self.horizontal_scale = horizontal_scale
        self.vertical_scale = vertical_scale
        self.u_off = u_off if u_off is not None else 0.0  # texture.rb:15-16
        self.v_off = v_off if v_off is not None else 0.0
        img = Image.open(self.file_name).convert("RGB")   # alpha ignored (:19)
        self.width, self.height = img.size                # columns, rows (:13-14)
        self.rgb8 = np.ascontiguousarray(np.asarray(img, dtype=np.uint8))  # [row][col][3]

    def texel_index(self, uu, vv):  # texture.rb:24-25 — trunc toward zero, then floored modulo
        u = int(math.trunc((uu + self.u_off) / self.horizontal_scale)) % self.width
        v = int(math.trunc((vv + self.v_off) / self.vertical_scale)) % self.height
        return u, v

    def to_a(self):
        return self.rgb8 / 256.0
