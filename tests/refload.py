"""Load the reference, kFYatek/color_modem, for golden generation and live cross-checks.

The reference is not part of this repository: set COLOR_MODEM_REFERENCE to the directory of a checkout (the one
holding the ``color_modem`` package).  Without it ``reference_available()`` is False and the tests that need it are
skipped.  Nothing here is used by the product.
"""
import contextlib
import os
import sys

import numpy as np

REFERENCE_ROOT = os.environ.get('COLOR_MODEM_REFERENCE', '')


def reference_available():
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, 'color_modem'))


class _Ref(object):
    pass


def _install_iirdesign_shim():
    """SURVEY.md §8c: scipy.signal.iirdesign without its wp/ws validation (same arithmetic otherwise)."""
    import scipy.signal
    from scipy.signal import _filter_design as fd
    if getattr(scipy.signal.iirdesign, '_cm_shim', False):
        return

    def iirdesign(wp, ws, gpass, gstop, analog=False, ftype='ellip', output='ba', fs=None):
        wp = np.atleast_1d(wp)
        ws = np.atleast_1d(ws)
        ordfunc = fd.filter_dict[ftype][1]
        band_type = 2 * (len(wp) - 1) + 1
        if wp[0] >= ws[0]:
            band_type += 1
        btype = {1: 'lowpass', 2: 'highpass', 3: 'bandstop', 4: 'bandpass'}[band_type]
        n, wn = ordfunc(wp, ws, gpass, gstop, analog=analog)
        return scipy.signal.iirfilter(n, wn, rp=gpass, rs=gstop, analog=analog, btype=btype, ftype=ftype,
                                      output=output)

    iirdesign._cm_shim = True
    scipy.signal.iirdesign = iirdesign


def load_reference():
    if not reference_available():
        raise RuntimeError('reference not present')
    sys.dont_write_bytecode = True
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    _install_iirdesign_shim()
    import color_modem.image as image
    import color_modem.line as line
    import color_modem.comb as comb
    from color_modem.color import ntsc, pal, secam, niir, protosecam, mac

    if not hasattr(ntsc.NtscVariant, 'NTSC_NOCOMB'):      # see oracle/presets.py
        ntsc.NtscVariant.NTSC_NOCOMB = ntsc.NtscVariant(fsc=227.0 * 15750.0 * 1000.0 / 1001.0)
    ref = _Ref()
    ref.image, ref.line, ref.comb = image, line, comb
    ref.ntsc, ref.pal, ref.secam, ref.niir, ref.protosecam, ref.mac = ntsc, pal, secam, niir, protosecam, mac

    def make_modem(c):
        std = getattr(line.LineStandard, c.standard) if c.standard else None
        lc = line.LineConfig((c.width, c.height), std)
        k, v = c.kind, c.variant
        notch = getattr(c, 'notch', 0.0)
        opt = getattr(c, 'opt', '')
        if k.startswith('scomb'):
            head, inner = k.split('+', 1)
            backend = make_modem(c._replace(kind=inner, notch=0.0, opt='', chroma_avg=False))
            m = comb.SimpleCombModem(backend, notch, comb.minavg if opt == 'minavg' else None, head == 'scomb3')
        elif k == 'ntsc':
            m = ntsc.NtscModem(lc, getattr(ntsc.NtscVariant, v))
        elif k == 'ntsc_comb':
            m = ntsc.NtscCombModem(lc, getattr(ntsc.NtscVariant, v), notch)
        elif k == 'ntsc_3d':
            m = comb.Simple3DCombModem(ntsc.NtscCombModem(lc, getattr(ntsc.NtscVariant, v)), notch,
                                       comb.minavg if opt == 'minavg' else None)
        elif k == 'pal_s':
            m = pal.PalSModem(lc, getattr(pal.PalVariant, v))
        elif k == 'pal_d':
            m = pal.PalDModem(lc, getattr(pal.PalVariant, v), notch)
        elif k == 'pal_3d':
            m = pal.Pal3DModem(lc, getattr(pal.PalVariant, v), notch, use_sin=(opt != 'nosin'), use_cos=(opt != 'nocos'),
                               avg=comb.minavg if opt == 'minavg' else None)
        elif k == 'secam':
            m = secam.SecamModem(lc, getattr(secam.SecamVariant, v), alternate_phases=(opt == 'altph'))
        elif k == 'niir':
            m = niir.NiirModem(lc, getattr(pal.PalVariant, v))
        elif k == 'niir_hue':
            m = niir.HueCorrectingNiirModem(lc, getattr(pal.PalVariant, v))
        elif k == 'protosecam':
            m = protosecam.ProtoSecamModem(lc, getattr(protosecam.ProtoSecamVariant, v), premod_luma_filter=(opt != 'noluma'))
        elif k == 'mac':
            m = mac.MacModem(lc, getattr(mac.MacVariant, v))
        else:
            raise ValueError(k)
        if c.chroma_avg:
            m = comb.ColorAveragingModem(m)
        return m

    @contextlib.contextmanager
    def capture_floats():
        """Record every float array the frame driver hands to image._as_bytes (image.py:54, 82)."""
        got = []
        orig = image._as_bytes

        def spy(a):
            got.append(np.array(a, dtype=np.float64))
            return orig(a)

        image._as_bytes = spy
        try:
            yield got
        finally:
            image._as_bytes = orig

    def rows_in_raster_order(got, height, per_row):
        """The driver emits field 0 (y=0,2,..) then field 1 (image.py:47,75); put rows back in raster order."""
        order = list(range(0, height, 2)) + list(range(1, height, 2))
        assert len(got) == per_row * height
        out = np.empty((height, per_row, len(got[0])), dtype=np.float64)
        for i, y in enumerate(order):
            for k in range(per_row):
                out[y, k] = got[i * per_row + k]
        return out

    ref.make_modem = make_modem
    ref.capture_floats = capture_floats
    ref.rows_in_raster_order = rows_in_raster_order
    return ref
