"""GPU-backed modem base: owns the native handles and implements both faces of the reference protocol.

* frame batches (the fast path, what ImageModem and bench.py use): ``encode_frames`` / ``decode_frames`` on
  CUDA ``torch.uint8`` tensors, or ``*_host`` on numpy arrays;
* the reference's per-line protocol ``modulate(frame, line, r, g, b)`` / ``demodulate(frame, line, composite)``
  (qam.py:68-72): float64 numpy rows in and out, with the same one-line memories and reset rule
  (``frame != last_frame or line != last_line + 2``, e.g. comb.py:48) as the reference's stateful classes.
  Each call gathers the neighbour rows it needs into a small row *window* and runs the same kernels on it.

torch is used only for device memory and streams.
"""
import ctypes as C

import numpy

from . import _native as N


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise N.NativeUnavailable('no CUDA device: color_modem_b200 has no CPU path')
    return torch


class GpuModem(object):
    """Base of every modem composition.  Subclasses provide ``_fill_desc(desc)`` and the row-window policy."""
    modulation_delay = 0
    demodulation_delay = 0

    def __init__(self, line_config, precision='fp32'):
        if precision not in ('fp32', 'fp64'):
            raise ValueError("precision must be 'fp32' or 'fp64'")
        self.line_config = line_config
        self.precision = precision
        if line_config.size[0] % 4:
            # the kernels move four samples per 32-bit / 128-bit access (include/color_modem_b200.h: cm_create)
            raise NotImplementedError('line widths must be multiples of 4 samples (got %d): the reference accepts any '
                                      'width, this implementation does not' % line_config.size[0])
        self._handles = {}
        self._enc_mem = None      # per-line protocol memories
        self._dec_mem = None

    # ---- geometry ----------------------------------------------------------------------------------------
    @property
    def width(self):
        return self.line_config.size[0]

    @property
    def height(self):
        return self.line_config.size[1]

    @property
    def composite_width(self):
        return self.width

    @property
    def output_width(self):
        return self.width

    # ---- native handle -----------------------------------------------------------------------------------
    def _base_desc(self):
        d = N.Desc()
        std = self.line_config.line_standard
        d.abi_version = N.ABI_VERSION
        d.width, d.height = self.width, self.height
        d.comp_width, d.out_width = self.composite_width, self.output_width
        d.digital_shift = self.line_config._line_shift
        d.odd_first = std.odd_field_first_active_line
        d.even_first = std.even_field_first_active_line
        d.ref_line = min(d.odd_first, d.even_first)
        d.frame_cycle = 1
        return d

    def describe(self):
        """The cm_desc handed to cm_create (pure host-side; usable without a GPU)."""
        d = self._base_desc()
        self._fill_desc(d)
        return d

    def _handle(self, precision=None, components=False):
        """Native handle of this composition.  ``components=True``: the same composition with identity colour matrices,
        i.e. the carrier of ``modulate_components`` / ``demodulate_components`` (planes in, planes out)."""
        precision = precision or self.precision
        key = (precision, bool(components))
        h = self._handles.get(key)
        if h is None:
            lib = N.load()
            _torch()
            desc = self.describe()
            if components:
                for i in range(9):
                    desc.enc_matrix[i] = desc.dec_matrix[i] = 1.0 if i % 4 == 0 else 0.0
            ptr = C.c_void_p()
            N.check(lib.cm_create(C.byref(desc), N.FP32 if precision == 'fp32' else N.FP64, C.byref(ptr)))
            h = self._handles[key] = ptr
        return h

    # ---- per-kernel device timing (bench.py roofline) ------------------------------------------------------
    def timing(self, on=True):
        N.check(N.load().cm_timing_enable(self._handle(), 1 if on else 0))
        N.check(N.load().cm_timing_reset(self._handle()))

    def timing_read(self, kernel_id):
        ms, n = C.c_double(0.0), C.c_int64(0)
        N.check(N.load().cm_timing_read(self._handle(), int(kernel_id), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def close(self):
        if self._handles:
            lib = N.load()
            for h in self._handles.values():
                lib.cm_destroy(h)
            self._handles = {}

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- frame batches on the device -----------------------------------------------------------------------
    def _check_outputs(self, src, out, out_float, tail):
        """out / out_float are written by the kernels through raw pointers: hold them to the exact layout."""
        torch = _torch()
        n = src.shape[0]
        for t, dtype in ((out, torch.uint8), (out_float, torch.float32 if self.precision == 'fp32' else torch.float64)):
            if t is None:
                continue
            if (not t.is_cuda or t.device != src.device or t.dtype != dtype or tuple(t.shape) != (n,) + tuple(tail)
                    or not t.is_contiguous()):
                raise ValueError('output must be a contiguous CUDA %s tensor of shape [%d, %s] on %s' % (
                    dtype, n, ', '.join(map(str, tail)), src.device))
            self._check_aligned(t)

    def encode_frames(self, rgb, first_frame=0, out=None, out_float=None):
        """rgb: CUDA uint8 tensor [N, H, W, 3] -> composite uint8 [N, H, Wc] (ImageModem.modulate, image.py:27-56)."""
        torch = _torch()
        self._check(rgb, torch.uint8, (self.height, self.width, 3))
        n = rgb.shape[0]
        self._check_outputs(rgb, out, out_float, (self.height, self.composite_width))
        if out is None and out_float is None:
            out = torch.empty((n, self.height, self.composite_width), dtype=torch.uint8, device=rgb.device)
        with torch.cuda.device(rgb.device):
            N.check(N.load().cm_encode_ex(self._handle(), None, rgb.data_ptr(), None,
                                          out.data_ptr() if out is not None else None,
                                          out_float.data_ptr() if out_float is not None else None,
                                          int(first_frame), int(n), torch.cuda.current_stream().cuda_stream))
        return out if out is not None else out_float

    def decode_frames(self, comp, first_frame=0, out=None, out_float=None):
        """comp: CUDA uint8 tensor [N, H, Wc] -> RGB uint8 [N, H, Wo, 3] (ImageModem.demodulate, image.py:58-84)."""
        torch = _torch()
        self._check(comp, torch.uint8, (self.height, self.composite_width))
        n = comp.shape[0]
        self._check_outputs(comp, out, out_float, (self.height, self.output_width, 3))
        if out is None and out_float is None:
            out = torch.empty((n, self.height, self.output_width, 3), dtype=torch.uint8, device=comp.device)
        with torch.cuda.device(comp.device):
            N.check(N.load().cm_decode_ex(self._handle(), None, comp.data_ptr(), None,
                                          out.data_ptr() if out is not None else None,
                                          out_float.data_ptr() if out_float is not None else None,
                                          int(first_frame), int(n), torch.cuda.current_stream().cuda_stream))
        return out if out is not None else out_float

    @staticmethod
    def _check(t, dtype, tail):
        if not t.is_cuda or t.dtype != dtype or tuple(t.shape[1:]) != tuple(tail) or not t.is_contiguous():
            raise ValueError('expected a contiguous CUDA %s tensor of shape [N, %s]' % (dtype, ', '.join(map(str, tail))))
        GpuModem._check_aligned(t)

    @staticmethod
    def _check_aligned(t):
        """The kernels move u8 frames in 32-bit words and float frames in vectors of four samples (16 bytes for float32,
        8-byte words for float64): a contiguous view at another storage offset is refused (include/color_modem_b200.h)."""
        torch = _torch()
        align = 4 if t.dtype == torch.uint8 else (16 if t.dtype == torch.float32 else 8)
        if t.numel() and t.data_ptr() % align:
            raise ValueError('frame buffer at %#x is not %d-byte aligned (a view at storage offset %d)' % (
                t.data_ptr(), align, t.storage_offset()))

    # ---- frame batches with host buffers (H2D + kernels + D2H inside the native call) ------------------------
    @staticmethod
    def _host_out(out, shape):
        if out is None:
            return numpy.empty(shape, dtype=numpy.uint8)
        if out.dtype != numpy.uint8 or out.shape != shape or not out.flags['C_CONTIGUOUS']:
            raise ValueError('out must be a C-contiguous uint8 array of shape %s' % (shape,))
        return out

    def _pic_in(self, pic, fmt, w):
        """Picture-side input batch: rgb24 [N, H, w, 3] or yuv420p [N, frame_bytes]."""
        from .pixfmt import frame_shape
        shape = frame_shape(fmt, w, self.height)
        pic = numpy.ascontiguousarray(pic, dtype=numpy.uint8)
        if pic.shape[1:] != shape:
            raise ValueError('expected %s uint8 [N, %s]' % (fmt.name, ', '.join(map(str, shape))))
        return pic

    def encode_frames_host(self, rgb, first_frame=0, out=None, pix_fmt=None):
        """rgb24 [N, H, W, 3] (or, with ``pix_fmt`` yuv420p, [N, frame_bytes]) host frames -> composite [N, H, Wc]."""
        from .pixfmt import resolve
        fmt = resolve(pix_fmt)
        rgb = self._pic_in(rgb, fmt, self.width)
        out = self._host_out(out, (rgb.shape[0], self.height, self.composite_width))
        if fmt.is_rgb24:
            N.check(N.load().cm_encode_frames_host(self._handle(), rgb.ctypes.data, out.ctypes.data, int(first_frame),
                                                   int(rgb.shape[0])))
        else:
            N.check(N.load().cm_encode_frames_host_fmt(self._handle(), rgb.ctypes.data, out.ctypes.data, int(first_frame),
                                                       int(rgb.shape[0]), C.byref(fmt.c_struct())))
        return out

    def decode_frames_host(self, comp, first_frame=0, out=None, pix_fmt=None):
        """composite [N, H, Wc] -> rgb24 [N, H, Wo, 3] (or, with ``pix_fmt`` yuv420p, [N, frame_bytes of Wo x H])."""
        from .pixfmt import frame_shape, resolve
        fmt = resolve(pix_fmt)
        comp = numpy.ascontiguousarray(comp, dtype=numpy.uint8)
        if comp.shape[1:] != (self.height, self.composite_width):
            raise ValueError('expected uint8 [N, %d, %d]' % (self.height, self.composite_width))
        out = self._host_out(out, (comp.shape[0],) + frame_shape(fmt, self.output_width, self.height))
        if fmt.is_rgb24:
            N.check(N.load().cm_decode_frames_host(self._handle(), comp.ctypes.data, out.ctypes.data, int(first_frame),
                                                   int(comp.shape[0])))
        else:
            N.check(N.load().cm_decode_frames_host_fmt(self._handle(), comp.ctypes.data, out.ctypes.data, int(first_frame),
                                                       int(comp.shape[0]), C.byref(fmt.c_struct())))
        return out

    def transcode_frames_host(self, rgb, first_frame=0, out=None, comp_out=None, want_composite=True, pix_fmt=None):
        """encode_frames_host followed by decode_frames_host of its result (what the reference's cli.py:62-65 does), the
        composite staying in device memory between the two.  Returns (composite or None, rgb).  With ``pix_fmt`` yuv420p
        both picture sides are yuv420p frames (the output ``output_width`` wide)."""
        from .pixfmt import frame_shape, resolve
        fmt = resolve(pix_fmt)
        rgb = self._pic_in(rgb, fmt, self.width)
        out = self._host_out(out, (rgb.shape[0],) + frame_shape(fmt, self.output_width, self.height))
        if want_composite or comp_out is not None:
            comp_out = self._host_out(comp_out, (rgb.shape[0], self.height, self.composite_width))
        comp_ptr = comp_out.ctypes.data if comp_out is not None else None
        if fmt.is_rgb24:
            N.check(N.load().cm_transcode_frames_host(self._handle(), rgb.ctypes.data, comp_ptr, out.ctypes.data,
                                                      int(first_frame), int(rgb.shape[0])))
        else:
            N.check(N.load().cm_transcode_frames_host_fmt(self._handle(), rgb.ctypes.data, comp_ptr, out.ctypes.data,
                                                          int(first_frame), int(rgb.shape[0]), C.byref(fmt.c_struct())))
        return comp_out, out

    # ---- float frames (parity tests: composite before the level map / RGB before clipping) -------------------
    def _np_dtype(self):
        return numpy.float32 if self.precision == 'fp32' else numpy.float64

    def _run_window(self, encode, frame, y0, rows_in, out_row, mode=N.MODE_DEFAULT, components=False, phase=0.0):
        """rows_in: float array [nrows, Win(, 3)] -> one output row as float64."""
        torch = _torch()
        dt = self._np_dtype()
        tin = torch.from_numpy(numpy.ascontiguousarray(rows_in, dtype=dt)).cuda()
        nrows = rows_in.shape[0]
        wout = self.composite_width if encode else self.output_width
        shape = (nrows, wout) if encode else (nrows, wout, 3)
        tout = torch.zeros(shape, dtype=tin.dtype, device=tin.device)
        from .utils import radians_fixed
        win = N.Window(nrows, int(y0), int(out_row), 1, int(mode), 0, radians_fixed(phase) if phase else 0)
        fn = N.load().cm_encode_ex if encode else N.load().cm_decode_ex
        N.check(fn(self._handle(components=components), C.byref(win), None, tin.data_ptr(), None, tout.data_ptr(),
                   int(frame), 1, torch.cuda.current_stream().cuda_stream))
        return tout[out_row].double().cpu().numpy()

    def encode_frame_float(self, rgb01, frame=0):
        """[H, W, 3] float RGB -> [H, Wc] composite as returned line by line by modem.modulate."""
        torch = _torch()
        tin = torch.from_numpy(numpy.ascontiguousarray(rgb01, dtype=self._np_dtype())).cuda()
        tout = torch.empty((self.height, self.composite_width), dtype=tin.dtype, device=tin.device)
        N.check(N.load().cm_encode_ex(self._handle(), None, None, tin.data_ptr(), None, tout.data_ptr(), int(frame), 1,
                                      torch.cuda.current_stream().cuda_stream))
        return tout.double().cpu().numpy()

    def decode_frame_float(self, comp, frame=0):
        """[H, Wc] float composite (after un-levelling) -> [H, Wo, 3] RGB as returned by modem.demodulate."""
        torch = _torch()
        tin = torch.from_numpy(numpy.ascontiguousarray(comp, dtype=self._np_dtype())).cuda()
        tout = torch.empty((self.height, self.output_width, 3), dtype=tin.dtype, device=tin.device)
        N.check(N.load().cm_decode_ex(self._handle(), None, None, tin.data_ptr(), None, tout.data_ptr(), int(frame), 1,
                                      torch.cuda.current_stream().cuda_stream))
        return tout.double().cpu().numpy()

    # ---- per-line protocol --------------------------------------------------------------------------------
    encoder_lookahead = False     # True: encoder reads the next line of the field (ColorAveraging / HueCorrecting)
    decoder_rows = 1              # 1: row itself; 2: + previous row; 3: previous, current and next (one-line delay)
    has_demodulate_components = False     # the reference class offers demodulate_components (comb-wrappable, SURVEY.md 8b)

    def _modulate_planes(self, frame, line, p0, p1, p2, components):
        cur = numpy.stack([numpy.asarray(p0, dtype=numpy.float64), numpy.asarray(p1, dtype=numpy.float64),
                           numpy.asarray(p2, dtype=numpy.float64)], axis=-1)
        if cur.shape[0] != self.width:
            raise AssertionError('line length does not match the modem width')
        if not self.encoder_lookahead:
            return self._run_window(True, frame, line, cur[None], 0, components=components)
        mem = self._enc_mem
        cont = mem is not None and mem[0] == frame and line == mem[1] + 2 and mem[3] == components
        self._enc_mem = (frame, line, cur, components)
        if not cont:      # comb.py:142-146 / niir.py:180-184: the line is paired with itself
            return self._run_window(True, frame, line - 2, cur[None], 0, components=components)
        rows = numpy.stack([mem[2], numpy.zeros_like(cur), cur])
        return self._run_window(True, frame, line - 2, rows, 0, components=components)

    def modulate(self, frame, line, r, g, b):
        """qam.py:68-69, secam.py:258, niir.py:76,176, protosecam.py:71, mac.py:124, comb.py:43,92,157."""
        return self._modulate_planes(frame, line, r, g, b, False)

    def modulate_components(self, frame, line, y, c1, c2):
        """ntsc.py:43-45, pal.py:48-52, secam.py:261, niir.py:80,179, protosecam.py:74, mac.py:42, comb.py:40,89,141:
        the same chain entered after the colour matrix (planes in the order of the class's encode_components)."""
        return self._modulate_planes(frame, line, y, c1, c2, True)

    def _demodulate_planes(self, frame, line, composite, components):
        cur = numpy.asarray(composite, dtype=numpy.float64)
        if len(cur) != self.composite_width:
            raise AssertionError('line length does not match the modem width')
        mem = self._dec_mem
        cont = mem is not None and mem[0] == frame and line == mem[1] + 2
        zero = numpy.zeros_like(cur)
        kw = {'components': components}
        if self.decoder_rows == 1:
            return cur, self._run_window(False, frame, line, cur[None], 0, **kw)
        if self.decoder_rows == 2:
            self._dec_mem = (frame, line, cur)
            if cont:
                return cur, self._run_window(False, frame, line - 2, numpy.stack([mem[2], zero, cur]), 2, **kw)
            return cur, self._run_window(False, frame, line, cur[None], 0, **kw)
        # one-line delay (Pal3DModem pal.py:180-234, Simple3DCombModem comb.py:96-113): the call for `line`
        # returns row line-2, computed from rows line-4 (if any), line-2 and line.
        if not cont:
            self._dec_mem = (frame, line, cur, None)
            return cur, self._run_window(False, frame, line, cur[None], 0, mode=N.MODE_BANDSPLIT_NOSTRIP, **kw)
        last, before = mem[2], mem[3]
        self._dec_mem = (frame, line, cur, last)
        if before is None:
            return last, self._run_window(False, frame, line - 2, numpy.stack([last, zero, cur]), 0, **kw)
        return last, self._run_window(False, frame, line - 4, numpy.stack([before, zero, last, zero, cur]), 2, **kw)

    def demodulate(self, frame, line, composite):
        """qam.py:71-72, comb.py:67-68,121-122, secam.py:278, niir.py:95, protosecam.py:92, mac.py:77."""
        _, rgb = self._demodulate_planes(frame, line, composite, False)
        return rgb[:, 0], rgb[:, 1], rgb[:, 2]

    def demodulate_components(self, frame, line, composite, strip_chroma=True):
        """ntsc.py:47-49, pal.py:54-59,180-234, comb.py:47-59, niir.py:98-163: (y, c1, c2) before the inverse matrix.
        strip_chroma=False leaves the luma un-stripped: the composite of the row the call answers for (the row itself, or
        the previous one for the decoders with a one-line delay); the chroma planes do not depend on the flag."""
        if not self.has_demodulate_components:
            raise AttributeError('%s has no demodulate_components (neither has the reference class)' % type(self).__name__)
        src, yuv = self._demodulate_planes(frame, line, composite, True)
        y = yuv[:, 0] if strip_chroma else numpy.array(src)
        return y, yuv[:, 1], yuv[:, 2]
