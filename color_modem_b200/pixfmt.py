"""Picture formats of the frame-batch paths: packed ``rgb24`` (the default everywhere) and planar 8-bit YUV 4:2:0
``yuv420p`` (I420), the format nearly every video file holds.

A ``yuv420p`` frame W x H is one row of ``frame_bytes`` bytes: the Y plane [H, W], then U (Cb) and V (Cr), each
[ceil(H/2), W/2].  Batches of such frames are [N, frame_bytes] uint8 arrays.  The conversion to and from RGB runs on the GPU
in exact integer arithmetic (Q16 coefficients derived from Kr, Kb and the range; INTEGRATION.md "Picture formats"):
RGB -> YUV averages each 2x2 chroma block (an odd height's last row counts twice), YUV -> RGB repeats each chroma sample over
its 2x2 block (nearest neighbour).  Nearest neighbour is deliberate: every modem's chroma low-pass (about 1.3 MHz for
PAL / NTSC) is far below the 3.4 MHz that 4:2:0 carries at 13.5 MHz, and the PAL-D, SECAM and MAC decoders average chroma
over two lines anyway, so the chroma siting variants (C420jpeg / mpeg2 / paldv) are all read the same way.
"""
import ctypes as C

from . import _native as N

NAMES = ('rgb24', 'yuv420p')
MATRICES = ('bt601', 'bt709')
RANGES = ('limited', 'full')


class PixelFormat(object):
    """``PixelFormat('yuv420p', matrix='bt601'|'bt709', range='limited'|'full')``; ``PixelFormat('rgb24')`` is the
    packed RGB of every existing call.  Defaults: BT.601, limited range (SD studio video)."""

    def __init__(self, name='rgb24', matrix='bt601', range='limited'):           # noqa: A002  (the ffmpeg / Y4M term)
        if name not in NAMES:
            raise ValueError('pixel format must be one of %s, not %r' % (', '.join(NAMES), name))
        if matrix not in MATRICES:
            raise ValueError('matrix must be one of %s, not %r' % (', '.join(MATRICES), matrix))
        if range not in RANGES:
            raise ValueError('range must be one of %s, not %r' % (', '.join(RANGES), range))
        self.name, self.matrix, self.range = name, matrix, range

    def __repr__(self):
        return 'PixelFormat(%r, matrix=%r, range=%r)' % (self.name, self.matrix, self.range)

    def __eq__(self, other):
        return isinstance(other, PixelFormat) and (self.name, self.matrix, self.range) == (other.name, other.matrix, other.range)

    def __hash__(self):
        return hash((self.name, self.matrix, self.range))

    @property
    def is_rgb24(self):
        return self.name == 'rgb24'

    def c_struct(self):
        return N.PixFmt(NAMES.index(self.name), MATRICES.index(self.matrix), RANGES.index(self.range), 0)


def resolve(pix_fmt):
    """None, a format name or a PixelFormat -> PixelFormat (None means rgb24)."""
    if pix_fmt is None:
        return PixelFormat('rgb24')
    if isinstance(pix_fmt, PixelFormat):
        return pix_fmt
    return PixelFormat(pix_fmt)


def frame_bytes(fmt, w, h):
    """Bytes of one frame w x h in format ``fmt``."""
    if resolve(fmt).is_rgb24:
        return w * h * 3
    return w * h + 2 * (w // 2) * ((h + 1) // 2)


def frame_shape(fmt, w, h):
    """Shape of one frame of a batch: (h, w, 3) for rgb24, (frame_bytes,) for yuv420p."""
    return (h, w, 3) if resolve(fmt).is_rgb24 else (frame_bytes(fmt, w, h),)


def _yuv_fmt(fmt):
    fmt = resolve(fmt)
    if fmt.is_rgb24:
        raise ValueError('the device conversions take a yuv420p PixelFormat')
    return fmt


def to_rgb24(yuv, fmt, w, h, out=None):
    """CUDA uint8 [N, frame_bytes(w, h)] yuv420p -> CUDA uint8 [N, h, w, 3] rgb24, on the current stream."""
    import torch
    fmt = _yuv_fmt(fmt)
    fb = frame_bytes(fmt, w, h)
    if not yuv.is_cuda or yuv.dtype != torch.uint8 or yuv.dim() != 2 or yuv.shape[1] != fb or not yuv.is_contiguous():
        raise ValueError('expected a contiguous CUDA uint8 tensor of shape [N, %d]' % fb)
    n = yuv.shape[0]
    if out is None:
        out = torch.empty((n, h, w, 3), dtype=torch.uint8, device=yuv.device)
    elif (not out.is_cuda or out.device != yuv.device or out.dtype != torch.uint8 or tuple(out.shape) != (n, h, w, 3)
          or not out.is_contiguous()):
        raise ValueError('out must be a contiguous CUDA uint8 tensor of shape [%d, %d, %d, 3] on %s' % (n, h, w, yuv.device))
    with torch.cuda.device(yuv.device):
        N.check(N.load().cm_yuv420p_to_rgb24(C.byref(fmt.c_struct()), yuv.data_ptr(), out.data_ptr(), int(w), int(h), int(n),
                                             torch.cuda.current_stream().cuda_stream))
    return out


def from_rgb24(rgb, fmt, out=None):
    """CUDA uint8 [N, H, W, 3] rgb24 -> CUDA uint8 [N, frame_bytes(W, H)] yuv420p, on the current stream."""
    import torch
    fmt = _yuv_fmt(fmt)
    if not rgb.is_cuda or rgb.dtype != torch.uint8 or rgb.dim() != 4 or rgb.shape[3] != 3 or not rgb.is_contiguous():
        raise ValueError('expected a contiguous CUDA uint8 tensor of shape [N, H, W, 3]')
    n, h, w = rgb.shape[0], rgb.shape[1], rgb.shape[2]
    fb = frame_bytes(fmt, w, h)
    if out is None:
        out = torch.empty((n, fb), dtype=torch.uint8, device=rgb.device)
    elif (not out.is_cuda or out.device != rgb.device or out.dtype != torch.uint8 or tuple(out.shape) != (n, fb)
          or not out.is_contiguous()):
        raise ValueError('out must be a contiguous CUDA uint8 tensor of shape [%d, %d] on %s' % (n, fb, rgb.device))
    with torch.cuda.device(rgb.device):
        N.check(N.load().cm_rgb24_to_yuv420p(C.byref(fmt.c_struct()), rgb.data_ptr(), out.data_ptr(), int(w), int(h), int(n),
                                             torch.cuda.current_stream().cuda_stream))
    return out
