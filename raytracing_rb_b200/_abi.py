"""ctypes mirror of include/rtrb_b200.h (structs, enums).  Layout must match the header field
for field; tests/test_abi.py checks sizeof() against the values the compiled library reports."""
import ctypes as C

ABI_VERSION = 4

RTRB_OK, RTRB_ERR_INVALID, RTRB_ERR_CUDA, RTRB_ERR_RAISED, RTRB_ERR_UNSUPPORTED = 0, 1, 2, 3, 4

ST_COLOR_GT_1 = 1 << 0
ST_ZERO_VECTOR = 1 << 1
ST_MATH_DOMAIN = 1 << 2
ST_STACK_OVERFLOW = 1 << 3
ST_NAN_TO_INT = 1 << 4

OBJ_PLANE, OBJ_SPHERE, OBJ_BOX = 0, 1, 2
FMT_RGBA8, FMT_RGB8, FMT_PNG_RGB8 = 0, 1, 2
RNG_CTR, RNG_MT = 0, 1
PREC_STRICT, PREC_FAST64 = 0, 1
PREC_DEFAULT = PREC_FAST64
SKIP_RGB, SKIP_HIT = 1, 2
PNG_SEGMENT_BYTES = 32768  # RTRB_PNG_SEGMENT_BYTES: the deflate segment of the device PNG encoder

D3 = C.c_double * 3


class ObjectDesc(C.Structure):
    _fields_ = [
        ("type", C.c_int32), ("texture", C.c_int32), ("has_refraction", C.c_int32), ("reserved0", C.c_int32),
        ("point", D3), ("radius", C.c_double),
        ("front", D3), ("up", D3),
        ("u_unit", C.c_double), ("v_unit", C.c_double),
        ("greenwich_vec", D3), ("north_pole_vec", D3),
        ("texture_horizontal_scale", C.c_double), ("texture_vertical_scale", C.c_double),
        ("texture_u_offset", C.c_double), ("texture_v_offset", C.c_double),
        ("refractive_rate", C.c_double),
        ("diffuse_rate", D3), ("reflective_attenuation", D3), ("refractive_attenuation", D3), ("ambient", D3),
        ("width_front", C.c_double), ("width_up", C.c_double), ("width_left", C.c_double),
    ]


class LightDesc(C.Structure):
    _fields_ = [
        ("position", D3), ("color", D3),
        ("radius", C.c_double), ("high_light_rate", C.c_double), ("high_light_angle", C.c_double),
    ]


class TextureDesc(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("rgb8", C.POINTER(C.c_uint8))]


class SceneDesc(C.Structure):
    _fields_ = [
        ("max_distance", C.c_double), ("soft_shadow_exponent", C.c_double),
        ("n_objects", C.c_int32), ("n_lights", C.c_int32), ("n_textures", C.c_int32), ("reserved0", C.c_int32),
        ("objects", C.POINTER(ObjectDesc)), ("lights", C.POINTER(LightDesc)), ("textures", C.POINTER(TextureDesc)),
    ]


class CameraDesc(C.Structure):
    _fields_ = [
        ("position", D3), ("up", D3), ("front", D3),
        ("retina_width", C.c_double), ("retina_height", C.c_double),
        ("aperture_radius", C.c_double), ("image_distance", C.c_double), ("focal_distance", C.c_double),
        ("variant_threshold", C.c_double),
        ("width", C.c_int32), ("height", C.c_int32),
        ("pre_sample_times", C.c_int32), ("max_sample_times", C.c_int32),
        ("trace_depth", C.c_int32), ("monte_carlo_diffusion_times", C.c_int32),
    ]


class RenderOpts(C.Structure):
    _fields_ = [
        ("rng_mode", C.c_int32), ("precision", C.c_int32), ("seed", C.c_uint64),
        ("x0", C.c_int32), ("y0", C.c_int32), ("x1", C.c_int32), ("y1", C.c_int32),
        ("tile_rank", C.c_int32), ("tile_world", C.c_int32),
        ("count_detail", C.c_int32), ("skip_outputs", C.c_int32),
        ("stream", C.c_void_p), ("rgba_device_out", C.c_void_p),
        ("pixel_format", C.c_int32), ("reserved0", C.c_int32),
    ]


class Ray(C.Structure):
    _fields_ = [("position", D3), ("front", D3)]


class RayHit(C.Structure):
    _fields_ = [
        ("object", C.c_int32), ("direction", C.c_int32), ("face", C.c_int32), ("reserved0", C.c_int32),
        ("distance", C.c_double), ("intersection", D3), ("delta", D3),
    ]


class RayOpts(C.Structure):
    _fields_ = [
        ("precision", C.c_int32), ("device_buffers", C.c_int32), ("seed", C.c_uint64),
        ("trace_depth", C.c_int32), ("monte_carlo_diffusion_times", C.c_int32),
        ("count_detail", C.c_int32),
        ("x0", C.c_int32), ("y0", C.c_int32), ("x1", C.c_int32), ("y1", C.c_int32),
        ("reserved0", C.c_int32),
        ("stream", C.c_void_p),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("samples", C.c_uint64), ("rays", C.c_uint64), ("shadow_queries", C.c_uint64),
        ("highlight_hits", C.c_uint64), ("hits", C.c_uint64), ("local_shaded", C.c_uint64),
        ("lit_lights", C.c_uint64), ("mc_rays", C.c_uint64), ("refractions", C.c_uint64),
        ("texel_fetches", C.c_uint64),
        ("sphere_tests", C.c_uint64), ("sphere_accepts", C.c_uint64),
        ("plane_tests", C.c_uint64), ("plane_accepts", C.c_uint64),
        ("cover_sphere", C.c_uint64), ("cover_sphere_full", C.c_uint64), ("cover_sphere_penumbra", C.c_uint64),
        ("cover_plane", C.c_uint64), ("cover_plane_accepts", C.c_uint64),
        ("adaptive_pixels", C.c_uint64), ("exact_tests", C.c_uint64),
        ("box_tests", C.c_uint64), ("box_accepts", C.c_uint64),
        ("cover_box", C.c_uint64), ("cover_box_accepts", C.c_uint64),
        ("status", C.c_uint32), ("first_bad_x", C.c_int32), ("first_bad_y", C.c_int32),
        ("max_stack", C.c_uint32), ("device_ms", C.c_float), ("trace_ms", C.c_float),
    ]

    COUNTER_FIELDS = (
        "samples", "rays", "shadow_queries", "highlight_hits", "hits", "local_shaded", "lit_lights", "mc_rays",
        "refractions", "texel_fetches", "sphere_tests", "sphere_accepts", "plane_tests", "plane_accepts",
        "cover_sphere", "cover_sphere_full", "cover_sphere_penumbra", "cover_plane", "cover_plane_accepts",
        "adaptive_pixels", "box_tests", "box_accepts", "cover_box", "cover_box_accepts",
    )

    def as_dict(self):
        d = {k: int(getattr(self, k)) for k in self.COUNTER_FIELDS}
        d.update(exact_tests=int(self.exact_tests), status=int(self.status), first_bad_x=int(self.first_bad_x),
                 first_bad_y=int(self.first_bad_y), max_stack=int(self.max_stack), device_ms=float(self.device_ms), trace_ms=float(self.trace_ms))
        return d
