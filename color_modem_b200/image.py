"""Frame-level driver — drop-in for ``color_modem.image.ImageModem`` (image.py:11-84).

``ImageModem(modem).modulate(img, frame)`` / ``.demodulate(img, frame)`` take and return PIL images exactly like
the reference.  The field-ordered line loop, delay priming and bottom-row wrap of image.py:47-55 / 75-83 are
folded into the kernels' row-window rules, so a frame is one native call (host->device copy, kernels,
device->host copy).  ``modulate_batch`` / ``demodulate_batch`` do the same for [N, H, W, C] uint8 arrays.
"""
import numpy


def _as_bytes(array):
    """image.py:7-8"""
    return numpy.uint8(numpy.rint(255.0 * numpy.maximum(numpy.minimum(array, 1.0), 0.0)))


def drive_demodulate_float(modem, composite, frame):
    """The line loop of image.py:75-83 over ``modem.demodulate`` for compositions that exist only as the per-line
    protocol (composed wrappers, comb.py): [H, Wc] float composite -> [H, Wo, 3] float RGB.  Every ``demodulate`` call
    runs on the GPU; this is the slow, general path — fused compositions never come here."""
    h = composite.shape[0]
    delay = getattr(modem, 'demodulation_delay', 0)
    rows = [None] * h
    for field in range(2):
        for y in range(field, 2 * delay, 2):
            if y < h:
                modem.demodulate(frame, y, composite[y])
        for y in range(field, h, 2):
            src = y + 2 * delay
            while src >= h:
                src -= 2
            rows[y] = numpy.stack(modem.demodulate(frame, y + 2 * delay, composite[src]), axis=-1)
    return numpy.stack(rows)


def drive_demodulate_u8(modem, comp_u8, frame):
    comp = ImageModem.decode_composite_level(numpy.asarray(comp_u8, dtype=numpy.uint8) / 255.0)
    return _as_bytes(drive_demodulate_float(modem, comp, frame))


class ImageModem(object):
    def __init__(self, modem):
        self._modem = modem

    @staticmethod
    def encode_composite_level(value):
        return 0.6 * value + 0.2

    @staticmethod
    def decode_composite_level(value):
        return (5.0 * value - 1.0) / 3.0

    def modulate_batch(self, rgb_u8, first_frame=0, out=None, pix_fmt=None):
        """[N, H, W, 3] rgb24 frames (or, with ``pix_fmt`` a yuv420p PixelFormat, [N, frame_bytes]) -> [N, H, Wc] composite."""
        return self._modem.encode_frames_host(rgb_u8, first_frame, out=out, pix_fmt=pix_fmt)

    def demodulate_batch(self, comp_u8, first_frame=0, out=None, pix_fmt=None):
        """[N, H, Wc] composite -> [N, H, Wo, 3] rgb24 frames (or [N, frame_bytes] yuv420p, ``output_width`` wide)."""
        return self._modem.decode_frames_host(comp_u8, first_frame, out=out, pix_fmt=pix_fmt)

    def transcode_batch(self, rgb_u8, first_frame=0, out=None, comp_out=None, want_composite=True, pix_fmt=None):
        """modulate_batch then demodulate_batch of the result in one native call: the composite is handed over in device
        memory (and copied out too unless ``want_composite`` is false).  Returns (composite or None, rgb).  With ``pix_fmt``
        yuv420p only the 4:2:0 frames cross the host link; the conversions run on the GPU."""
        return self._modem.transcode_frames_host(rgb_u8, first_frame, out=out, comp_out=comp_out,
                                                 want_composite=want_composite, pix_fmt=pix_fmt)

    def modulate(self, img, frame=0):
        from PIL import Image
        if img.mode != 'RGB':
            img = img.convert('RGB')
        rgb = numpy.asarray(img, dtype=numpy.uint8)
        comp = self.modulate_batch(rgb[None], frame)[0]
        return Image.fromarray(comp, 'L')

    def demodulate(self, img, frame=0):
        from PIL import Image
        if img.mode != 'L':
            img = img.convert('L')
        comp = numpy.asarray(img, dtype=numpy.uint8)
        rgb = self.demodulate_batch(comp[None], frame)[0]
        return Image.fromarray(rgb, 'RGB')
