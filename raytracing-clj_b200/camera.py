"""Camera derivation, host side, IEEE double, in the reference's operation order.

Follows (does not copy) the three `-main` let-blocks of the reference:
  main   src/raytracing.clj:105-139
  realm  src/realm/raytracing.clj:20-26, 264-280, 306-322
  -i     src/experimental/raytracing_i.clj:82-90, 127-144
Python floats are IEEE doubles and CPython never fuses a*b+c, so every vector below
is what the JVM computes, up to the last bit of Math/tan (a <=1-ulp libm function on
both sides; SURVEY.md 8c).  The native twin of this file is rtclj_camera_* in
csrc/host.cpp; tests/test_host.py checks they agree bit for bit.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from decimal import Context, Decimal, ROUND_HALF_EVEN
from fractions import Fraction
from typing import Sequence, Tuple

Vec = Tuple[float, float, float]

_DECIMAL64 = Context(prec=16, rounding=ROUND_HALF_EVEN)


def ratio_to_double(num: int, den: int) -> float:
    """What Clojure yields when the exact rational num/den meets a double.

    `(/ 400 225)` is the Ratio 16/9; Ratio.doubleValue divides as BigDecimal under
    MathContext.DECIMAL64 (16 significant digits) and converts that decimal, which is
    one ulp ABOVE 16.0/9.0 (SURVEY.md Appendix B.1; corroborated by the 400x224
    header of the reference's scene-realm.ppm).  Integral quotients stay exact."""
    fr = Fraction(num, den)
    if fr.denominator == 1:
        return float(fr.numerator)
    return float(_DECIMAL64.divide(Decimal(fr.numerator), Decimal(fr.denominator)))


def image_height_main(width: int, aspect: Fraction = Fraction(16, 9)) -> int:
    """raytracing.clj:107 -- exact rational division, then `int` (truncate)."""
    return int(Fraction(width) / aspect)


def image_height_realm(width: int, aspect: Fraction = Fraction(16, 9)) -> int:
    """realm/raytracing.clj:22 and raytracing_i.clj:82-84 -- double division by the
    Ratio's double value: 400 / 1.777777777777778 = 224.99999999999997 -> 224."""
    return int(float(width) / ratio_to_double(aspect.numerator, aspect.denominator))


def _sub(a: Vec, b: Vec) -> Vec:
    return (a[0] - b[0], a[1] - b[1], a[2] - b[2])


def _add(a: Vec, b: Vec) -> Vec:
    return (a[0] + b[0], a[1] + b[1], a[2] + b[2])


def _muls(a: Vec, s: float) -> Vec:
    return (a[0] * s, a[1] * s, a[2] * s)


def _divs(a: Vec, s: float) -> Vec:
    return (a[0] / s, a[1] / s, a[2] / s)


def _neg(a: Vec) -> Vec:
    return (-a[0], -a[1], -a[2])


def _cross(u: Vec, v: Vec) -> Vec:  # vec3a.clj:64-67
    return (u[1] * v[2] - u[2] * v[1], u[2] * v[0] - u[0] * v[2], u[0] * v[1] - u[1] * v[0])


def _length(a: Vec) -> float:  # vec3a.clj:56-59
    return math.sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2])


def _unit(a: Vec) -> Vec:  # vec3a.clj:69
    return _divs(a, _length(a))


def deg_to_rad(d: float) -> float:  # raytracing.clj:60-61
    return d * math.pi / 180.0


@dataclass
class Camera:
    """The values that cross the C ABI (rtclj_camera in include/rtclj_b200.h)."""

    width: int
    height: int
    pixel00: Vec
    pixel_du: Vec
    pixel_dv: Vec
    center: Vec
    defocus_u: Vec = (0.0, 0.0, 0.0)
    defocus_v: Vec = (0.0, 0.0, 0.0)
    defocus_angle: float = 0.0
    meta: dict = field(default_factory=dict)


def main_camera(
    width: int = 400,
    height: int | None = None,
    vfov: float = 20.0,
    look_from: Sequence[float] = (-2.0, 2.0, 1.0),
    look_at: Sequence[float] = (0.0, 0.0, -1.0),
    vup: Sequence[float] = (0.0, 1.0, 0.0),
    defocus_angle: float = 10.0,
    focus_dist: float = 3.4,
) -> Camera:
    """raytracing.clj:105-139 (defaults are its literals)."""
    if height is None:
        height = image_height_main(width)
    look_from, look_at, vup = tuple(map(float, look_from)), tuple(map(float, look_at)), tuple(map(float, vup))
    theta = deg_to_rad(vfov)
    h = math.tan(theta / 2)
    viewport_height = 2.0 * h * focus_dist
    viewport_width = viewport_height * ratio_to_double(width, height)
    w = _unit(_sub(look_from, look_at))
    u = _unit(_cross(vup, w))
    v = _cross(w, u)
    center = look_from
    viewport_u = _muls(u, viewport_width)
    viewport_v = _muls(_neg(v), viewport_height)
    pixel_du = _divs(viewport_u, float(width))
    pixel_dv = _divs(viewport_v, float(height))
    upper_left = _sub(_sub(_sub(center, _muls(w, focus_dist)), _divs(viewport_u, 2.0)), _divs(viewport_v, 2.0))
    pixel00 = _add(upper_left, _muls(_add(pixel_du, pixel_dv), 0.5))
    defocus_radius = focus_dist * math.tan(deg_to_rad(defocus_angle / 2.0))
    return Camera(
        width, height, pixel00, pixel_du, pixel_dv, center,
        _muls(u, defocus_radius), _muls(v, defocus_radius), float(defocus_angle),
        {"variant": "main", "u": u, "v": v, "w": w},
    )


def turntable_look_from(k: int, n: int, look_from: Sequence[float] = (-2.0, 2.0, 1.0),
                        look_at: Sequence[float] = (0.0, 0.0, -1.0)) -> tuple:
    """look_from rotated by k * 360/n degrees about the vertical axis through look_at (frame k of an n-frame
    turntable); k = 0 is look_from itself."""
    look_from, look_at = tuple(map(float, look_from)), tuple(map(float, look_at))
    if k % n == 0:
        return look_from
    a = 2.0 * math.pi * k / n
    dx, dz = look_from[0] - look_at[0], look_from[2] - look_at[2]
    return (look_at[0] + dx * math.cos(a) + dz * math.sin(a), look_from[1], look_at[2] - dx * math.sin(a) + dz * math.cos(a))


def turntable_cameras(n: int, width: int = 400, height: int | None = None) -> list:
    """The reference's main camera on an n-frame turntable around its look_at: frame 0 is main_camera()."""
    return [main_camera(width, height, look_from=turntable_look_from(k, n)) for k in range(n)]


def realm_camera(
    width: int = 400,
    height: int | None = None,
    vfov: float = 20.0,
    look_from: Sequence[float] = (-2.0, 2.0, 1.0),
    look_at: Sequence[float] = (0.0, 0.0, -1.0),
    vup: Sequence[float] = (0.0, 1.0, 0.0),
) -> Camera:
    """realm/raytracing.clj:264-280, 306-322: focus distance = |look-from - look-at|,
    no defocus, aspect = W/H as doubles."""
    if height is None:
        height = image_height_realm(width)
    look_from, look_at, vup = tuple(map(float, look_from)), tuple(map(float, look_at)), tuple(map(float, vup))
    temp = _sub(look_from, look_at)
    focal = _length(temp)
    w = _divs(temp, focal)
    u = _unit(_cross(vup, w))
    v = _cross(w, u)
    theta = deg_to_rad(vfov)
    h = math.tan(theta / 2.0)
    viewport_height = 2.0 * h * focal
    viewport_width = viewport_height * (float(width) / float(height))
    viewport_u = _muls(u, viewport_width)
    viewport_v = _muls(v, -viewport_height)
    pixel_du = _divs(viewport_u, float(width))
    pixel_dv = _divs(viewport_v, float(height))
    ul = _sub(look_from, _muls(w, focal))
    ul = _sub(ul, _divs(viewport_u, 2.0))
    ul = _sub(ul, _divs(viewport_v, 2.0))
    pixel00 = _add(ul, _divs(_add(pixel_du, pixel_dv), 2.0))
    return Camera(width, height, pixel00, pixel_du, pixel_dv, look_from,
                  meta={"variant": "realm", "u": u, "v": v, "w": w})


def i_camera(width: int = 400, height: int | None = None) -> Camera:
    """experimental/raytracing_i.clj:82-90, 127-144: camera at the origin looking
    down -z, focal length 1, viewport height 2."""
    if height is None:
        height = image_height_realm(width)
    focal_length = 1.0
    viewport_height = 2.0
    viewport_width = viewport_height * ratio_to_double(width, height)
    center = (0.0, 0.0, 0.0)
    viewport_u = (viewport_width, 0.0, 0.0)
    viewport_v = (0.0, -viewport_height, 0.0)
    pixel_du = _divs(viewport_u, float(width))
    pixel_dv = _divs(viewport_v, float(height))
    ul = _sub(center, (0.0, 0.0, focal_length))
    ul = _sub(ul, _divs(viewport_u, 2.0))
    ul = _sub(ul, _divs(viewport_v, 2.0))
    pixel00 = _add(ul, _divs(_add(pixel_du, pixel_dv), 2.0))
    return Camera(width, height, pixel00, pixel_du, pixel_dv, center, meta={"variant": "i"})
