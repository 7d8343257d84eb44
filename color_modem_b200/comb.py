"""Line-memory wrappers — drop-in for ``color_modem.comb`` (comb.py:9-167).

The reference composes decoders at run time out of Python objects that call each other line by line.  Here a
composition is served in one of two ways:

* **fused**: the compositions the reference's own driver script lists as its decoders of choice are single kernel
  families — ``Simple3DCombModem(NtscCombModem(lc))`` (cli.py:24) is the 3-line NTSC comb, ``ColorAveragingModem(x)``
  (cli.py:40,44,56) switches on the look-ahead chroma averaging inside the encoder kernel of ``x``;
* **composed**: every other legal composition — ``SimpleCombModem`` / ``Simple3DCombModem`` over any backend that offers
  ``demodulate_components`` (NtscModem, PalSModem, NtscCombModem, PalDModem, Pal3DModem, NiirModem,
  HueCorrectingNiirModem, another wrapper ...), e.g. cli.py:52 — runs the reference's line-by-line protocol with every
  backend call (demodulation, re-modulation through the backend's encoder, luma notch) executed by the backend's CUDA
  kernels on a row window.  That path is exact but launches several small kernels per line: it exists for completeness
  of the drop-in, not for throughput (the reference's own comment on cli.py:52: "turned out to be a bad idea").

There is no CPU fallback: without the CUDA library every compute call raises NativeUnavailable.
"""
import numpy

from . import _native as N
from . import utils


def avg(val1, val2):
    """comb.py:9-10"""
    return 0.5 * (val1 + val2)


def minavg(val1, val2):
    """comb.py:13-15: the smaller magnitude where the two estimates agree in sign, zero where they do not"""
    sign = (1.0 - numpy.signbit(val1)) - numpy.signbit(val2)
    return sign * numpy.minimum(numpy.abs(val1), numpy.abs(val2))


def _is_reference_fn(fn, name):
    """True for color_modem.comb.<name> of an installed reference (so a drop-in caller may pass the reference's own)."""
    return getattr(fn, '__module__', None) == 'color_modem.comb' and getattr(fn, '__name__', None) == name


def _avg_mode(fn):
    """Which of the reference's two combiners `fn` is: False = mean (None or comb.avg), True = comb.minavg.
    Matched by identity (this module's functions or the reference module's), never by bare name."""
    if fn is None or fn is avg or _is_reference_fn(fn, 'avg'):
        return False
    if fn is minavg or _is_reference_fn(fn, 'minavg'):
        return True
    raise NotImplementedError('avg= accepts comb.avg or comb.minavg; arbitrary Python callables cannot run in the kernels')


def _notch(qam_modem, q):
    """comb.py:18-20"""
    import scipy.signal
    b, a = scipy.signal.iirnotch(2.0 * qam_modem.config.fsc / qam_modem.line_config.fs, q)
    return utils.FilterFunction(b, a, wp=0.0, btype='bandstop', shift=True)


def _clone(backend, **changes):
    """A re-configured copy of a GpuModem (own native handles, own line memories)."""
    m = object.__new__(type(backend))
    m.__dict__.update(backend.__dict__)
    m._handles = {}
    m._enc_mem = m._dec_mem = None
    if getattr(backend, 'backend', None) is backend:
        m.backend = m
    for k, v in changes.items():
        setattr(m, k, v)
    return m


def _fp64_twin(modem):
    """The same composition with float64 kernels.  Composed wrappers run every backend call through it: the path is bound
    by launches, not arithmetic, and the NIIR backends (hue from atan2 after the saturation clamp of niir.py:61-65) are
    discontinuous at zero chroma, where float32 rounding would decide the hue."""
    from .modem import GpuModem
    if isinstance(modem, GpuModem):
        return modem if modem.precision == 'fp64' else _clone(modem, precision='fp64')
    impl = getattr(modem, '_impl', None)
    if impl is not None:
        twin = object.__new__(type(modem))
        twin.__dict__.update(modem.__dict__)
        twin._impl = _fp64_twin(impl)
        return twin
    return modem          # a composed wrapper: already float64 inside


def _gpu_impl(modem):
    """The GpuModem that does the work of `modem` (a GpuModem itself, or a fused wrapper around one); None for composed
    wrappers."""
    from .modem import GpuModem
    if isinstance(modem, GpuModem):
        return modem
    return getattr(modem, '_impl', None)


class _Fused(object):
    """Delegates the protocol to a re-configured clone of the backend."""
    _impl = None

    config = property(lambda self: self.backend.config)
    line_config = property(lambda self: self.backend.line_config)
    modulation_delay = property(lambda self: self._impl.modulation_delay)
    demodulation_delay = property(lambda self: self._impl.demodulation_delay)

    def __getattr__(self, name):          # encode_frames, decode_frames, modulate, demodulate, describe, ...
        if name.startswith('_'):           # never recurse on a half-built instance (copy.copy, pickling)
            raise AttributeError(name)
        impl = self.__dict__.get('_impl')
        if impl is None:
            raise AttributeError(name)
        return getattr(impl, name)


class SimpleCombModem(_Fused):
    """comb.py:71-122.  Averages the chroma of consecutive lines of a field as decoded by ``backend`` and subtracts its
    re-modulation from the luma; ``delay=True`` centres the pair on the output line (one line of decoding delay)."""

    def __init__(self, backend, notch=0.0, avg=None, delay=False):
        self.backend = backend
        self._own_delay = 1 if delay else 0
        self._minavg = _avg_mode(avg)
        self._avg = minavg if self._minavg else globals()['avg']
        self._notch_q = float(notch)
        self._last_frame = -1
        self._last_line = -1
        self._last_demodulated = None
        self._impl = None
        self._notch = None
        from .color.ntsc import NtscCombModem
        if delay and type(backend) is NtscCombModem and numpy.isfinite(backend._factor):
            # the wrapper's own notch (comb.py:108-109); the backend's is never applied (it is called with strip_chroma=False)
            self._impl = _clone(backend, kind=N.KIND_NTSC_3D, decoder_rows=3, _notch_q=self._notch_q, _minavg=self._minavg,
                                demodulation_delay=getattr(backend, 'demodulation_delay', 0) + 1)
            return
        if not hasattr(backend, 'demodulate_components') or not getattr(backend, 'has_demodulate_components', True):
            raise AttributeError('%s has no demodulate_components: not comb-wrappable (as in the reference)'
                                 % type(backend).__name__)
        self._exec = _fp64_twin(backend)
        self._modulation_delay = getattr(backend, 'modulation_delay', 0)
        self._demodulation_delay = getattr(backend, 'demodulation_delay', 0) + self._own_delay
        if self._notch_q:
            self._notch = _notch(backend, self._notch_q)

    modulation_delay = property(lambda self: self._impl.modulation_delay if self._impl else self._modulation_delay)
    demodulation_delay = property(lambda self: self._impl.demodulation_delay if self._impl else self._demodulation_delay)
    has_demodulate_components = True

    # ---- composed path: the reference's state machine over GPU backend calls --------------------------------
    def modulate_components(self, frame, line, y, u, v):
        return self.backend.modulate_components(frame, line, y, u, v)

    def modulate(self, frame, line, r, g, b):
        return self.backend.modulate(frame, line, r, g, b)

    def encode_components(self, r, g, b):
        return self.backend.encode_components(r, g, b)

    def decode_components(self, y, u, v):
        return self.backend.decode_components(y, u, v)

    def _precision(self):
        impl = _gpu_impl(self.backend)
        return getattr(impl, 'precision', None) or getattr(self.backend, 'precision', 'fp32')

    precision = property(_precision)

    def demodulate_components(self, frame, line, composite, strip_chroma=True):
        if self._impl is not None:
            return self._impl.demodulate_components(frame, line, composite, strip_chroma)
        curr = self._exec.demodulate_components(frame, line, composite, strip_chroma=False)
        if frame != self._last_frame or line != self._last_line + 2:
            y, u, v = curr
        else:
            last = self._last_demodulated
            y = last[0] if self._own_delay else curr[0]
            u = self._avg(last[1], curr[1])
            v = self._avg(last[2], curr[2])
            if strip_chroma:
                y = y - self._exec.modulate_components(frame, line - 2 * (self._own_delay - self._modulation_delay),
                                                       numpy.zeros(len(composite)), u, v)
                if self._notch is not None:
                    y = self._notch(y, precision='fp64')
        self._last_frame = frame
        self._last_line = line
        self._last_demodulated = curr
        return y, u, v

    def demodulate(self, frame, line, composite):
        if self._impl is not None:
            return self._impl.demodulate(frame, line, composite)
        return self.backend.decode_components(*self.demodulate_components(frame, line, composite))

    # ---- frame batches --------------------------------------------------------------------------------------
    def encode_frames(self, rgb, first_frame=0, out=None, out_float=None):
        return (self._impl or self.backend).encode_frames(rgb, first_frame, out=out, out_float=out_float)

    def encode_frames_host(self, rgb, first_frame=0, out=None, pix_fmt=None):
        return (self._impl or self.backend).encode_frames_host(rgb, first_frame, out=out, pix_fmt=pix_fmt)

    def decode_frames_host(self, comp, first_frame=0, out=None, pix_fmt=None):
        if self._impl is not None:
            return self._impl.decode_frames_host(comp, first_frame, out=out, pix_fmt=pix_fmt)
        from .image import drive_demodulate_u8
        from .pixfmt import from_rgb24, frame_shape, resolve
        fmt = resolve(pix_fmt)
        comp = numpy.ascontiguousarray(comp, dtype=numpy.uint8)
        res = numpy.stack([drive_demodulate_u8(self, comp[i], first_frame + i) for i in range(comp.shape[0])]) \
            if comp.shape[0] else numpy.empty((0, comp.shape[1], self.backend.output_width, 3), numpy.uint8)
        if not fmt.is_rgb24:          # the composed path is u8 RGB; the conversion runs on the device around it
            import torch
            res = from_rgb24(torch.from_numpy(res).cuda(), fmt).cpu().numpy() if res.shape[0] else \
                numpy.empty((0,) + frame_shape(fmt, self.backend.output_width, comp.shape[1]), numpy.uint8)
        if out is not None:
            out[...] = res
            return out
        return res

    def transcode_frames_host(self, rgb, first_frame=0, out=None, comp_out=None, want_composite=True, pix_fmt=None):
        if self._impl is not None:
            return self._impl.transcode_frames_host(rgb, first_frame, out=out, comp_out=comp_out,
                                                    want_composite=want_composite, pix_fmt=pix_fmt)
        comp = self.encode_frames_host(rgb, first_frame, out=comp_out, pix_fmt=pix_fmt)
        return (comp if want_composite or comp_out is not None else None), \
            self.decode_frames_host(comp, first_frame, out=out, pix_fmt=pix_fmt)

    def decode_frames(self, comp, first_frame=0, out=None, out_float=None):
        if self._impl is not None:
            return self._impl.decode_frames(comp, first_frame, out=out, out_float=out_float)
        if out_float is not None:
            raise NotImplementedError('composed wrappers return u8 frames only')
        import torch
        res = torch.from_numpy(self.decode_frames_host(comp.cpu().numpy(), first_frame)).to(comp.device)
        if out is not None:
            out.copy_(res)
            return out
        return res

    def encode_frame_float(self, rgb01, frame=0):
        return (self._impl or self.backend).encode_frame_float(rgb01, frame)

    def decode_frame_float(self, comp, frame=0):
        if self._impl is not None:
            return self._impl.decode_frame_float(comp, frame)
        from .image import drive_demodulate_float
        return drive_demodulate_float(self, numpy.asarray(comp, dtype=numpy.float64), frame)

    def describe(self):
        """cm_desc of the kernels that serve this composition (the fused kind, or the backend's for the composed path)."""
        return (self._impl or self.backend).describe()

    width = property(lambda self: self.backend.width)
    height = property(lambda self: self.backend.height)
    composite_width = property(lambda self: self.backend.composite_width)
    output_width = property(lambda self: self.backend.output_width)


class Simple3DCombModem(SimpleCombModem):
    """comb.py:125-127"""

    def __init__(self, backend, notch=0.0, avg=None):
        super(Simple3DCombModem, self).__init__(backend, notch, avg, True)


class ColorAveragingModem(_Fused):
    """Encoder-side averaging of each line's chroma with the next line of the field (comb.py:130-167)."""

    def __init__(self, backend):
        self.backend = backend
        inner = _gpu_impl(backend)
        if inner is None:
            raise NotImplementedError('ColorAveragingModem over a composed wrapper is not built')
        if getattr(inner, 'encoder_lookahead', False):
            raise NotImplementedError('ColorAveragingModem over a look-ahead encoder is not a reference composition')
        base_flags = inner._flags

        def flags():
            return base_flags() | N.FLAG_CHROMA_AVG

        self._impl = _clone(inner, _flags=flags, encoder_lookahead=True,
                            modulation_delay=getattr(inner, 'modulation_delay', 0) + 1)
