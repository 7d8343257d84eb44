"""Planar YUV 4:2:0 (I420) <-> packed RGB24, restated in numpy from the integer definition (test infrastructure).

The coefficients are derived here from the rule itself, not read from the product:

* matrices: bt601 Kr = 0.299, Kb = 0.114; bt709 Kr = 0.2126, Kb = 0.0722; Kg = 1 - Kr - Kb;
* ranges: limited Y' = 16 + 219 E'y, C = 128 + 224 E'c; full Y' = 255 E'y, C = 128 + 255 E'c;
* Q16 fixed point, each coefficient round_half_away(2^16 * value); the forward chroma G coefficients make each chroma row
  sum to 0, the forward luma G coefficient makes the luma row sum to round(2^16 * s) (s = 219/255 or 1);
* RGB -> YUV: Y' = (cYR R + cYG G + cYB B + oY 2^16 + 2^15) >> 16; Cb / Cr sum the unrounded products over the 2x2 block and
  round once, (S + 128 2^18 + 2^17) >> 18; an odd height's last row stands in for the missing row of its block;
* YUV -> RGB: chroma upsampled by nearest neighbour, R = (cY (Y' - oY) + cRV (Cr - 128) + 2^15) >> 16 and likewise G, B.

Shifts are arithmetic (floor); results are clipped to [0, 255].
"""
import math

import numpy

MATRICES = {'bt601': (0.299, 0.114), 'bt709': (0.2126, 0.0722)}
RANGES = ('limited', 'full')


def round_half_away(x):
    return int(math.copysign(math.floor(abs(x) + 0.5), x))


def coefficients(matrix='bt601', rng='limited'):
    """dict of the Q16 integer coefficients of one matrix / range set."""
    kr, kb = MATRICES[matrix]
    kg = 1.0 - kr - kb
    limited = rng == 'limited'
    if rng not in RANGES:
        raise ValueError(rng)
    sy = 219.0 / 255.0 if limited else 1.0
    sc = 224.0 / 255.0 if limited else 1.0
    q = 65536.0
    c = {'oY': 16 if limited else 0}
    c['YR'] = round_half_away(q * sy * kr)
    c['YB'] = round_half_away(q * sy * kb)
    c['YG'] = round_half_away(q * sy) - c['YR'] - c['YB']
    c['UR'] = round_half_away(q * sc * -kr / (2.0 * (1.0 - kb)))
    c['UB'] = round_half_away(q * sc * 0.5)
    c['UG'] = -(c['UR'] + c['UB'])
    c['VR'] = round_half_away(q * sc * 0.5)
    c['VB'] = round_half_away(q * sc * -kb / (2.0 * (1.0 - kr)))
    c['VG'] = -(c['VR'] + c['VB'])
    iy = 255.0 / 219.0 if limited else 1.0
    ic = 255.0 / 224.0 if limited else 1.0
    c['Y'] = round_half_away(q * iy)
    c['RV'] = round_half_away(q * ic * 2.0 * (1.0 - kr))
    c['GU'] = round_half_away(q * ic * -2.0 * kb * (1.0 - kb) / kg)
    c['GV'] = round_half_away(q * ic * -2.0 * kr * (1.0 - kr) / kg)
    c['BU'] = round_half_away(q * ic * 2.0 * (1.0 - kb))
    return c


def frame_bytes(w, h):
    return w * h + 2 * (w // 2) * ((h + 1) // 2)


def split_planes(frames, w, h):
    """[N, frame_bytes] -> Y [N, H, W], U [N, ceil(H/2), W/2], V [N, ceil(H/2), W/2] (views)."""
    n, hc, wc = frames.shape[0], (h + 1) // 2, w // 2
    y = frames[:, :w * h].reshape(n, h, w)
    u = frames[:, w * h:w * h + wc * hc].reshape(n, hc, wc)
    v = frames[:, w * h + wc * hc:].reshape(n, hc, wc)
    return y, u, v


def rgb_to_yuv420p(rgb, matrix='bt601', rng='limited'):
    """rgb uint8 [N, H, W, 3] -> uint8 [N, frame_bytes]."""
    c = coefficients(matrix, rng)
    rgb = numpy.asarray(rgb, dtype=numpy.int64)
    n, h, w, _ = rgb.shape
    r, g, b = rgb[..., 0], rgb[..., 1], rgb[..., 2]
    y = (c['YR'] * r + c['YG'] * g + c['YB'] * b + c['oY'] * 65536 + 32768) >> 16
    pu = c['UR'] * r + c['UG'] * g + c['UB'] * b
    pv = c['VR'] * r + c['VG'] * g + c['VB'] * b
    if h % 2:                                   # the last row stands in for the missing one
        pu = numpy.concatenate([pu, pu[:, -1:]], axis=1)
        pv = numpy.concatenate([pv, pv[:, -1:]], axis=1)

    def block(p):
        s = p[:, 0::2, 0::2] + p[:, 0::2, 1::2] + p[:, 1::2, 0::2] + p[:, 1::2, 1::2]
        return (s + 128 * (1 << 18) + (1 << 17)) >> 18

    out = numpy.empty((n, frame_bytes(w, h)), numpy.uint8)
    oy, ou, ov = split_planes(out, w, h)
    oy[...] = numpy.clip(y, 0, 255)
    ou[...] = numpy.clip(block(pu), 0, 255)
    ov[...] = numpy.clip(block(pv), 0, 255)
    return out


def yuv420p_to_rgb(frames, w, h, matrix='bt601', rng='limited'):
    """uint8 [N, frame_bytes] -> rgb uint8 [N, H, W, 3] (nearest-neighbour chroma)."""
    c = coefficients(matrix, rng)
    frames = numpy.asarray(frames, dtype=numpy.uint8)
    y, u, v = split_planes(frames, w, h)
    y = y.astype(numpy.int64) - c['oY']
    u = numpy.repeat(numpy.repeat(u.astype(numpy.int64) - 128, 2, axis=1), 2, axis=2)[:, :h]
    v = numpy.repeat(numpy.repeat(v.astype(numpy.int64) - 128, 2, axis=1), 2, axis=2)[:, :h]
    ly = c['Y'] * y + 32768
    r = (ly + c['RV'] * v) >> 16
    g = (ly + c['GU'] * u + c['GV'] * v) >> 16
    b = (ly + c['BU'] * u) >> 16
    return numpy.clip(numpy.stack([r, g, b], axis=-1), 0, 255).astype(numpy.uint8)
