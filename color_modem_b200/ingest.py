"""Batched frame ingest: raw packed video files <-> the batch entry points (SURVEY.md §8 f3).

The reference opens and saves one PIL image per frame (cli.py:19,62,64).  Here frame sequences are read as packed raw
video — ``rgb24`` ([N, H, W, 3] bytes, what ``ffmpeg -f rawvideo -pix_fmt rgb24`` writes), ``yuv420p`` (planar 4:2:0,
``-pix_fmt yuv420p``, as a raw ``.yuv`` file or as YUV4MPEG2 ``.y4m``) and ``gray8`` composite ([N, H, Wc]) — straight into
pinned host buffers that the native host entry points copy from: a reader thread fills batch i+1 and a
writer thread drains batch i-1 while batch i is on the GPU (whose own three-stream pipeline overlaps its copies with the
kernels).  No per-frame Python objects, no PIL on this path.
"""
import os
import queue
import threading

import numpy


def _pinned(shape):
    """uint8 array in page-locked memory when torch + CUDA are there (the copies then run at link speed), plain otherwise."""
    try:
        import torch
        if torch.cuda.is_available():
            return torch.empty(shape, dtype=torch.uint8).pin_memory().numpy()
    except Exception:                                                   # noqa: BLE001
        pass
    return numpy.empty(shape, dtype=numpy.uint8)


class RawVideo(object):
    """A file of packed frames of ``frame_shape`` bytes each (``(H, W, 3)`` for rgb24, ``(frame_bytes,)`` for yuv420p,
    ``(H, W)`` for gray8), after a file header of ``header`` bytes, each frame preceded by the constant ``prefix`` (Y4M:
    the file header line and ``FRAME\n``).  Frame i starts at ``header + i * (len(prefix) + frame_bytes)``."""

    def __init__(self, path, frame_shape, mode='r', header=0, prefix=b''):
        self.path, self.frame_shape = path, tuple(int(v) for v in frame_shape)
        self.frame_bytes = int(numpy.prod(self.frame_shape))
        self.header, self.prefix = int(header), bytes(prefix)
        self.stride = len(self.prefix) + self.frame_bytes
        self._f = open(path, 'rb' if mode == 'r' else ('r+b' if os.path.exists(path) and mode == 'a' else 'wb'))
        self.nframes = max(0, os.path.getsize(path) - self.header) // self.stride if mode == 'r' else 0

    def read_into(self, first, out):
        """Frames [first, first + len(out)) into ``out`` (a C-contiguous uint8 array); returns the number read."""
        if not self.prefix:
            self._f.seek(self.header + first * self.frame_bytes)
            got = self._f.readinto(memoryview(out).cast('B'))
            return got // self.frame_bytes
        for i in range(len(out)):
            self._f.seek(self.header + (first + i) * self.stride)
            p = self._f.read(len(self.prefix))
            if len(p) < len(self.prefix):
                return i
            if p != self.prefix:
                raise ValueError('%s: frame %d does not start with %r (frame headers with parameters are not supported: '
                                 'frames are found by their offset)' % (self.path, first + i, self.prefix))
            if self._f.readinto(memoryview(out[i]).cast('B')) < self.frame_bytes:
                return i
        return len(out)

    def write_at(self, first, frames):
        frames = numpy.ascontiguousarray(frames)
        self._f.seek(self.header + first * self.stride)
        if self.prefix:
            buf = numpy.empty((len(frames), self.stride), numpy.uint8)
            buf[:, :len(self.prefix)] = numpy.frombuffer(self.prefix, numpy.uint8)
            buf[:, len(self.prefix):] = frames.reshape(len(frames), -1)
            frames = buf
        self._f.write(memoryview(frames).cast('B'))

    def write_header(self, data):
        self._f.seek(0)
        self._f.write(data)

    def close(self):
        self._f.close()


Y4M_MAGIC = b'YUV4MPEG2'
Y4M_FRAME = b'FRAME\n'
Y4M_420 = ('420', '420jpeg', '420mpeg2', '420paldv')      # 4:2:0 siting variants, all read the same way (pixfmt.py)


def is_y4m(path):
    return os.path.splitext(path)[1].lower() == '.y4m'


def is_yuv(path):
    """A path whose extension names yuv420p frames: raw ``.yuv`` or ``.y4m``."""
    return os.path.splitext(path)[1].lower() in ('.yuv', '.y4m')


def picture_paths(op, src_path, dst_path):
    """The paths of ``op`` that hold pictures (the others hold the gray8 composite)."""
    return [p for p, pic in ((src_path, op != 'demodulate'), (dst_path, op != 'modulate')) if pic and p]


def read_y4m_header(path):
    """The header line of a Y4M file, ``\n`` included."""
    with open(path, 'rb') as f:
        head = f.read(4096)
    end = head.find(b'\n')
    if not head.startswith(Y4M_MAGIC + b' ') or end < 0:
        raise ValueError('%s: not a YUV4MPEG2 file' % path)
    return head[:end + 1]


def parse_y4m_header(header):
    """dict(width, height, chroma, range) of a Y4M header line; range is 'full', 'limited' or None (not stated).
    Only 8-bit 4:2:0 is accepted (C420, C420jpeg, C420mpeg2, C420paldv; no C tag means C420jpeg)."""
    tokens = header.rstrip(b'\n').split(b' ')
    if tokens[0] != Y4M_MAGIC:
        raise ValueError('not a YUV4MPEG2 header')
    info = {'width': None, 'height': None, 'chroma': '420jpeg', 'range': None}
    for t in tokens[1:]:
        t = t.decode('ascii', 'replace')
        if t.startswith('W'):
            info['width'] = int(t[1:])
        elif t.startswith('H'):
            info['height'] = int(t[1:])
        elif t.startswith('C'):
            info['chroma'] = t[1:]
        elif t.startswith('XCOLORRANGE='):
            v = t[len('XCOLORRANGE='):].upper()
            if v not in ('FULL', 'LIMITED'):
                raise ValueError('Y4M XCOLORRANGE=%s: FULL or LIMITED expected' % v)
            info['range'] = v.lower()
    if info['width'] is None or info['height'] is None:
        raise ValueError('Y4M header without W / H')
    if info['chroma'] not in Y4M_420:
        raise ValueError('Y4M colour space C%s is not supported: 8-bit 4:2:0 only (C420, C420jpeg, C420mpeg2, C420paldv)'
                         % info['chroma'])
    return info


def y4m_with_width(header, width):
    """The header line with its W token set to ``width`` (MAC decodes to 720 samples whatever the input width)."""
    tokens = header.rstrip(b'\n').split(b' ')
    return b' '.join(b'W%d' % width if t.startswith(b'W') else t for t in tokens) + b'\n'


def y4m_header(width, height, frame_rate, fmt):
    """Header of a Y4M output written without a Y4M input to copy it from."""
    from fractions import Fraction
    fr = Fraction(frame_rate).limit_denominator(1001)
    return b'YUV4MPEG2 W%d H%d F%d:%d Ip A1:1 C420jpeg XCOLORRANGE=%s\n' % (
        width, height, fr.numerator, fr.denominator, fmt.range.upper().encode())


def picture_format(path, fmt):
    """The format of a picture-side input file: ``fmt`` (a PixelFormat) for raw files; for Y4M yuv420p with the file's
    XCOLORRANGE, when stated, in place of ``fmt.range``."""
    from .pixfmt import PixelFormat
    if not is_y4m(path):
        return fmt
    info = parse_y4m_header(read_y4m_header(path))
    return PixelFormat('yuv420p', fmt.matrix, info['range'] or fmt.range)


def open_source(modem, op, path, fmt):
    """RawVideo of the input of ``op`` (gray8 composite for demodulate, picture frames in ``fmt`` otherwise)."""
    from .pixfmt import frame_shape
    if op == 'demodulate':
        return RawVideo(path, (modem.height, modem.composite_width))
    shape = frame_shape(fmt, modem.width, modem.height)
    if not is_y4m(path):
        return RawVideo(path, shape)
    header = read_y4m_header(path)
    info = parse_y4m_header(header)
    if (info['width'], info['height']) != (modem.width, modem.height):
        raise ValueError('%s is %dx%d, the modem %dx%d' % (path, info['width'], info['height'], modem.width, modem.height))
    return RawVideo(path, shape, header=len(header), prefix=Y4M_FRAME)


def output_header(modem, op, src_path, dst_path, fmt):
    """The file header of the picture output ``dst_path``: b'' unless it is Y4M; then the input's header with W set to
    ``output_width`` when the input is Y4M too, a fresh one otherwise."""
    if op == 'modulate' or not is_y4m(dst_path):
        return b''
    if op == 'transcode' and is_y4m(src_path):
        return y4m_with_width(read_y4m_header(src_path), modem.output_width)
    return y4m_header(modem.output_width, modem.height, modem.line_config.line_standard.frame_rate, fmt)


def frame_batches(first, last, batch):
    return [(b, min(b + batch, last)) for b in range(first, last, batch)]


def run_file(modem, op, src_path, dst_path, dst2_path=None, first_frame=0, frames=None, batch=64, out_offset=None,
             pix_fmt=None):
    """Stream a raw video file through ``modem``.

    op = 'modulate'   picture -> gray8 composite            (dst)
         'demodulate' gray8 composite -> picture            (dst)
         'transcode'  picture -> picture decoded (dst) and, if dst2_path is given, the gray8 composite (dst2)
    Pictures are ``pix_fmt`` frames (a PixelFormat; None = rgb24); a ``.y4m`` path is a YUV4MPEG2 file of yuv420p frames
    (its XCOLORRANGE, when stated, sets the range).  A Y4M output gets the input's header (W = ``output_width``), or a
    fresh one, unless the file already holds a header.  The composite is always raw gray8.
    Frame i of the file is absolute frame i (carrier phase and line parity depend on it).  ``frames`` = (a, b) restricts
    the run to file frames [a, b); they are written at the same positions of the outputs (``out_offset`` shifts them),
    so several processes — one per GPU, each with its own contiguous range — can fill one output file.
    Returns the number of frames processed."""
    from .image import ImageModem
    from .pixfmt import PixelFormat, frame_shape, resolve
    img = ImageModem(modem)
    fmt = resolve(pix_fmt)
    if fmt.is_rgb24 and any(is_yuv(p) for p in picture_paths(op, src_path, dst_path)):
        fmt = PixelFormat('yuv420p', fmt.matrix, fmt.range)
    if op != 'demodulate':
        fmt = picture_format(src_path, fmt)
    h, wc, wo = modem.height, modem.composite_width, modem.output_width
    out_shape = (h, wc) if op == 'modulate' else frame_shape(fmt, wo, h)
    src = open_source(modem, op, src_path, fmt)
    in_shape = src.frame_shape
    pic_fmt = None if fmt.is_rgb24 else fmt
    a, b = (0, src.nframes) if frames is None else (max(0, frames[0]), min(src.nframes, frames[1]))
    shift = -a if out_offset is None else out_offset - a
    header = output_header(modem, op, src_path, dst_path, fmt)
    dst = RawVideo(dst_path, out_shape, 'a', header=len(header), prefix=Y4M_FRAME if header else b'')
    if header and os.path.getsize(dst_path) < len(header):
        dst.write_header(header)
    dst2 = RawVideo(dst2_path, (h, wc), 'a') if (op == 'transcode' and dst2_path) else None
    ring = 3
    bufs_in = [_pinned((batch,) + in_shape) for _ in range(ring)]
    bufs_out = [_pinned((batch,) + out_shape) for _ in range(ring)]
    bufs_mid = [_pinned((batch, h, wc)) for _ in range(ring)] if dst2 else [None] * ring
    free, filled, done = queue.Queue(), queue.Queue(), queue.Queue()
    for i in range(ring):
        free.put(i)
    err = []

    def reader():
        try:
            for lo, hi in frame_batches(a, b, batch):
                i = free.get()
                n = src.read_into(lo, bufs_in[i][:hi - lo])
                filled.put((i, lo, n))
        except Exception as e:                                           # noqa: BLE001
            err.append(e)
        filled.put(None)

    def writer():
        try:
            while True:
                item = done.get()
                if item is None:
                    break
                i, lo, n = item
                dst.write_at(lo + shift, bufs_out[i][:n])
                if dst2:
                    dst2.write_at(lo + shift, bufs_mid[i][:n])
                free.put(i)
        except Exception as e:                                           # noqa: BLE001
            err.append(e)

    tr, tw = threading.Thread(target=reader), threading.Thread(target=writer)
    tr.start()
    tw.start()
    total = 0
    try:
        while True:
            item = filled.get()
            if item is None or err:
                break
            i, lo, n = item
            if n:
                if op == 'modulate':
                    img.modulate_batch(bufs_in[i][:n], first_frame + lo, out=bufs_out[i][:n], pix_fmt=pic_fmt)
                elif op == 'demodulate':
                    img.demodulate_batch(bufs_in[i][:n], first_frame + lo, out=bufs_out[i][:n], pix_fmt=pic_fmt)
                else:
                    img.transcode_batch(bufs_in[i][:n], first_frame + lo, out=bufs_out[i][:n],
                                        comp_out=bufs_mid[i][:n] if dst2 else None, want_composite=bool(dst2),
                                        pix_fmt=pic_fmt)
            total += n
            done.put((i, lo, n))
    finally:
        done.put(None)
        tr.join()
        tw.join()
        src.close()
        dst.close()
        if dst2:
            dst2.close()
    if err:
        raise err[0]
    return total
