"""cv2-free integer model of the reference sampler + single-pass per-pixel restatement.
TEST INFRASTRUCTURE (see ``oracle/__init__.py``).

Two things live here:

* ``remap_fixedpoint`` - what ``cv2.remap(src, U, V, INTER_LINEAR, BORDER_CONSTANT)`` computes
  for 8-bit images (the call at ref ``app/panorama_to_plane-pitch.py:192-199`` and ``:212-218``).
  The arithmetic lives in the third-party dependency ``opencv-python`` (pinned 4.10.0.84 in the
  reference's ``requirements.txt:13``; 4.13.0 in this image) and is not vendored under
  ``/root/reference``; its published algorithm (``modules/imgproc/src/imgwarp.cpp``:
  ``remap`` -> ``convertMaps`` to ``CV_16SC2`` + 5-bit fraction index -> ``remapBilinear`` with
  ``FixedPtCast<int, uchar, INTER_REMAP_COEF_BITS=15>``) is restated here:
      sx = round_half_even(U * 32)  (f32 multiply), ix = sx >> 5, fx = sx & 31  (same for y)
      out = (p00*(32-fx)*(32-fy) + p01*fx*(32-fy) + p10*(32-fx)*fy + p11*fx*fy + 512) >> 10
  with out-of-image taps reading the constant border 0 and NaN coordinates landing far outside
  the image (-> 0).  The real tables hold ``saturate_cast<short>((1-fy)(1-fx) * 32768)`` etc.;
  for a 32x32 fraction grid those are exact multiples of 32 and the table fix-up is a no-op, so
  ``(sum + 2^14) >> 15`` equals the 10-bit form above.  ``tests/test_oracle_golden.py`` checks the
  model against real ``cv2.remap`` on random maps, and against the stored reference outputs.

* ``project_view_single_pass`` - the per-output-pixel restatement the CUDA kernel implements
  (SURVEY.md Appendix A): coordinates from the pitch map, the yaw pass folded in as a
  panorama-column lookup (``yaw_column_table``), one integer blend.  Bit-identical to the
  two-pass reference whenever the yaw column table has no fractional part (every yaw with
  ``yaw * Wp / 360`` integral); the general case goes through ``apply_yaw_table`` first, exactly
  like the reference's yaw ``cv2.remap``.
"""
from __future__ import annotations

import numpy as np

from . import ref_port

INTER_BITS = 5
INTER_TAB = 1 << INTER_BITS  # 32


def quantise(coord: np.ndarray):
    """f32 map -> (integer part, 5-bit fraction, nan mask) the way cv::remap's convertMaps does.

    ``cvRound(x * 32)`` with an f32 product, round-half-even.  NaN converts to INT_MIN
    (cvtps2dq) which lands outside any image; we return an explicit mask instead.
    """
    coord = np.asarray(coord, dtype=np.float32)
    nan = np.isnan(coord)
    scaled = np.where(nan, np.float32(0), coord) * np.float32(INTER_TAB)
    s = np.rint(scaled).astype(np.int64)
    return s >> INTER_BITS, s & (INTER_TAB - 1), nan


def remap_fixedpoint(src: np.ndarray, U: np.ndarray, V: np.ndarray) -> np.ndarray:
    """Integer model of ``cv2.remap(src, U, V, INTER_LINEAR, BORDER_CONSTANT(0))`` for u8 images."""
    src = np.asarray(src)
    assert src.dtype == np.uint8 and src.ndim == 3
    Hs, Ws, _ = src.shape
    ix, fx, nx = quantise(U)
    iy, fy, ny = quantise(V)
    dead = nx | ny

    def tap(yy, xx):
        inside = (xx >= 0) & (xx < Ws) & (yy >= 0) & (yy < Hs) & ~dead
        px = src[np.clip(yy, 0, Hs - 1), np.clip(xx, 0, Ws - 1)].astype(np.int64)
        return px * inside[..., None]

    w00 = ((INTER_TAB - fx) * (INTER_TAB - fy))[..., None]
    w01 = (fx * (INTER_TAB - fy))[..., None]
    w10 = ((INTER_TAB - fx) * fy)[..., None]
    w11 = (fx * fy)[..., None]
    acc = (
        tap(iy, ix) * w00 + tap(iy, ix + 1) * w01 + tap(iy + 1, ix) * w10 + tap(iy + 1, ix + 1) * w11
    )
    return ((acc + (1 << (2 * INTER_BITS - 1))) >> (2 * INTER_BITS)).astype(np.uint8)


# ---------------------------------------------------------------------------------------------
# yaw pass as a column table
# ---------------------------------------------------------------------------------------------
def yaw_column_table(pano_width: int, yaw_deg):
    """(ix, fx) per rotated column: the quantised form of one row of the reference yaw map
    (ref :95-105; rows are identical because V = v, :102)."""
    ix, fx, nan = quantise(ref_port.yaw_row(pano_width, yaw_deg))
    assert not nan.any()
    return ix.astype(np.int32), fx.astype(np.int32)


def yaw_table_is_roll(ix: np.ndarray, fx: np.ndarray):
    """Return the integer column shift if the table is a pure roll ``ix[u] = (u + shift) % Wp``
    with no fractional part, else None."""
    Wp = ix.shape[0]
    if fx.any():
        return None
    shift = int(ix[0])
    if np.array_equal(ix, (np.arange(Wp, dtype=np.int64) + shift) % Wp):
        return shift
    return None


def apply_yaw_table(pano: np.ndarray, ix: np.ndarray, fx: np.ndarray) -> np.ndarray:
    """The reference's yaw ``cv2.remap`` (:192-199) in integer form: fy = 0, so
    ``rot[v,u] = (p[v,ix]*(32-fx) + p[v,ix+1]*fx + 16) >> 5`` (tap ix+1 == Wp only ever has fx = 0
    because of the clip at :105)."""
    Wp = pano.shape[1]
    a = pano[:, ix].astype(np.int64)
    b = pano[:, np.minimum(ix + 1, Wp - 1)].astype(np.int64)
    b = b * (ix + 1 < Wp)[None, :, None]
    f = fx.astype(np.int64)[None, :, None]
    return ((a * (INTER_TAB - f) + b * f + 16) >> INTER_BITS).astype(np.uint8)


# ---------------------------------------------------------------------------------------------
# exact f32 fused multiply-add on f32 arrays (what the sgemm inner loop does, SURVEY App. A step 3)
# ---------------------------------------------------------------------------------------------
def fma32(a, b, c):
    """Correctly rounded f32 ``a*b + c`` for f32 inputs.

    The product of two f32 is exact in f64; the f64 sum may round, so it is re-rounded to odd
    (sticky bit) before the final conversion to f32, which makes the double rounding harmless.
    """
    a = np.asarray(a, np.float32).astype(np.float64)
    b = np.asarray(b, np.float32).astype(np.float64)
    c = np.asarray(c, np.float32).astype(np.float64)
    p = a * b
    s = p + c
    # TwoSum error term (exact)
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    inexact = (err != 0) & np.isfinite(s)
    bits = s.view(np.int64).copy()
    # truncate toward zero: if the error points toward zero, step one ulp toward zero
    toward_zero = inexact & ((err < 0) == (s > 0)) & (s != 0)
    bits = np.where(toward_zero, bits - 1, bits)
    bits = np.where(inexact, bits | 1, bits)
    return bits.view(np.float64).astype(np.float32)


def pitch_coords_scalar_model(W, H, fov_deg, pitch_deg, Wp, Hp, rows=None):
    """Per-pixel op sequence of SURVEY Appendix A steps 1-5 (what the CUDA kernel executes),
    with NumPy's own f32 ``arccos`` / ``arctan2`` for the two transcendentals.

    Unlike ``ref_port.pitch_mapping`` this does not call sgemm: the rotation is the explicit
    k-ordered FMA chain.  ``tests/test_oracle_golden.py`` asserts it equals the reference map
    bit for bit on this host.  ``rows``: compute only these output rows (maps of shape
    [len(rows), W]), for views too large to map whole.
    """
    f, c, s = ref_port.pitch_scalars(W, fov_deg, pitch_deg)
    u = np.arange(W, dtype=np.float32)[None, :]
    v = (np.arange(H) if rows is None else np.asarray(rows)).astype(np.float32)[:, None]
    shape = (v.shape[0], W)
    x = np.broadcast_to(u - np.float32(W / 2.0), shape)
    y = np.broadcast_to(np.float32(H / 2.0) - v, shape)
    z = np.full(shape, f, dtype=np.float32)
    n = np.sqrt((x * x + y * y) + z * z)
    xn, yn, zn = x / n, y / n, z / n
    zero = np.float32(0) * xn
    x_rot = fma32(np.float32(0), zn, fma32(np.float32(0), yn, fma32(np.float32(1), xn, np.float32(0))))
    y_rot = fma32(-s, zn, fma32(c, yn, zero + np.float32(0)))
    z_rot = fma32(c, zn, fma32(s, yn, zero + np.float32(0)))
    with np.errstate(invalid="ignore"):
        theta = np.arccos(z_rot)
    a = np.arctan2(y_rot, x_rot)
    two_pi = np.float32(2 * np.pi)
    phi = np.where(a < 0, a + two_pi, a).astype(np.float32)
    U = (phi * np.float32(Wp)) / two_pi
    V = (theta * np.float32(Hp)) / np.float32(np.pi)
    U = np.clip(U, 0, Wp - 1).astype(np.float32)
    V = np.clip(V, 0, Hp - 1).astype(np.float32)
    return U, V


def sample_view(pano, U, V, yaw_ix=None, yaw_shift=None):
    """Single-pass sampler: quantised pitch coordinates, yaw folded in as a column lookup
    (integer roll) and the 4-tap integer blend.  SURVEY Appendix A steps 6-8."""
    Hp, Wp, _ = pano.shape
    ix, fx, nx = quantise(U)
    iy, fy, ny = quantise(V)
    dead = nx | ny
    if yaw_ix is None:
        yaw_ix = (np.arange(Wp, dtype=np.int64) + int(yaw_shift or 0)) % Wp
    ix0 = np.clip(ix, 0, Wp - 1)
    ix1 = np.clip(ix + 1, 0, Wp - 1)
    iy0 = np.clip(iy, 0, Hp - 1)
    iy1 = np.clip(iy + 1, 0, Hp - 1)
    c0 = yaw_ix[ix0]
    c1 = yaw_ix[ix1]

    def p(yy, xx):   # gather first: the taps, not the whole panorama, are widened to int64
        return pano[yy, xx].astype(np.int64)

    wx0, wy0 = (INTER_TAB - fx)[..., None], (INTER_TAB - fy)[..., None]
    wx1, wy1 = fx[..., None], fy[..., None]
    acc = p(iy0, c0) * wx0 * wy0 + p(iy0, c1) * wx1 * wy0 + p(iy1, c0) * wx0 * wy1 + p(iy1, c1) * wx1 * wy1
    out = ((acc + 512) >> 10).astype(np.uint8)
    out[dead] = 0
    return out


def project_view_single_pass(pano, yaw_deg, pitch_deg, W, H, fov_deg=90, coords=None):
    """One view the way the CUDA path computes it.  ``coords`` lets a test inject (U, V)."""
    Hp, Wp, _ = pano.shape
    if coords is None:
        coords = ref_port.pitch_mapping(W, H, fov_deg, pitch_deg, Wp, Hp)
    ix, fx = yaw_column_table(Wp, yaw_deg)
    if yaw_table_is_roll(ix, fx) is not None:
        return sample_view(pano, coords[0], coords[1], yaw_ix=ix.astype(np.int64))
    rotated = apply_yaw_table(pano, ix, fx)
    return sample_view(rotated, coords[0], coords[1], yaw_shift=0)


def touched_texels(pano_shape, views, W, H, fov_deg):
    """N_T of SURVEY section 8(d): number of distinct panorama texels that receive a non-zero
    bilinear weight in at least one of ``views`` = [(yaw_deg, pitch_deg), ...]."""
    Hp, Wp = pano_shape[:2]
    mask = np.zeros((Hp, Wp), dtype=bool)
    for yaw, pitch in views:
        U, V = ref_port.pitch_mapping(W, H, fov_deg, pitch, Wp, Hp)
        ix, fx, nx = quantise(U)
        iy, fy, ny = quantise(V)
        ok = ~(nx | ny)
        yix, yfx = yaw_column_table(Wp, yaw)
        assert not yfx.any()
        for dy, wy in ((0, INTER_TAB - fy), (1, fy)):
            for dx, wx in ((0, INTER_TAB - fx), (1, fx)):
                sel = ok & (wy * wx > 0)
                yy = np.clip(iy + dy, 0, Hp - 1)[sel]
                xx = yix[np.clip(ix + dx, 0, Wp - 1)[sel]]
                mask[yy, xx] = True
    return int(mask.sum())
