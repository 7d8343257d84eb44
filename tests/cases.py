"""Golden-vector case list shared by tests/golden/make_golden.py and the parity tests.

Each case names a reference composition (oracle ``kind``), preset, raster and absolute frame index.
Frames are small (24 rows) with an explicit line standard so the fixtures stay a few MB in total;
``LineConfig((W, 24), standard)`` is a legal reference configuration (line.py:50-55).
"""
import collections
import hashlib
import os

import numpy as np

Case = collections.namedtuple('Case', 'kind variant width height standard chroma_avg frame seed content notch opt')
# notch: Q of the luma notch of the comb decoders (comb.py:18-20), 0 = off
# opt:   other non-default constructor knobs: 'nosin' / 'nocos' (Pal3DModem use_sin / use_cos = False, pal.py:131),
#        'altph' (SecamModem alternate_phases=True, secam.py:163-166), 'noluma' (ProtoSecamModem premod_luma_filter=False),
#        'minavg' (Simple3DCombModem / Pal3DModem avg=comb.minavg, comb.py:13-15)
Case.__new__.__defaults__ = (0.0, '')


def _c(kind, variant, std, frame, width=720, height=24, avg=False, seed=None, content='smooth', notch=0.0, opt=''):
    return Case(kind, variant, width, height, std, avg, frame, frame * 7 + 1 if seed is None else seed, content, notch,
                opt)


GOLDEN_CASES = [
    # NTSC family (ntsc.py, comb.py)
    _c('ntsc', 'NTSC', 'NTSC_525', 0),
    _c('ntsc_comb', 'NTSC', 'NTSC_525', 1),
    _c('ntsc_3d', 'NTSC', 'NTSC_525', 2),
    _c('ntsc_3d', 'NTSC443', 'NTSC_525', 7),
    _c('ntsc', 'NTSC361', 'NTSC_525', 3, content='noise'),
    _c('ntsc_comb', 'NTSC_A', 'BAIRD_405', 4),
    _c('ntsc', 'NTSC_I', 'GERBER_625', 5),
    _c('ntsc_comb', 'NTSC_N', 'GERBER_625', 6),
    # PAL family (pal.py)
    _c('pal_s', 'PAL', 'GERBER_625', 0),
    _c('pal_d', 'PAL', 'GERBER_625', 1),
    _c('pal_d', 'PAL', 'GERBER_625', 2, content='noise'),
    _c('pal_3d', 'PAL', 'GERBER_625', 3),
    _c('pal_d', 'PAL_M', 'NTSC_525', 5),
    _c('pal_s', 'PAL_M', 'NTSC_525', 2),
    _c('pal_3d', 'PAL_N', 'GERBER_625', 6),
    # SECAM (secam.py) incl. ColorAveragingModem encoder (comb.py:130-167)
    _c('secam', 'SECAM', 'GERBER_625', 0),
    _c('secam', 'SECAM', 'GERBER_625', 1, avg=True),
    _c('secam', 'SECAM', 'GERBER_625', 4, content='noise'),
    _c('secam', 'SECAM_I', 'GERBER_625', 2),
    _c('secam', 'SECAM_II', 'GERBER_625', 3),
    _c('secam', 'SECAM_III', 'GERBER_625', 5),
    _c('secam', 'SECAM_A', 'BAIRD_405', 2),
    _c('secam', 'SECAM_M', 'NTSC_525', 3),
    _c('secam', 'SECAM_N', 'GERBER_625', 4),
    # NIIR / SECAM-IV (niir.py)
    _c('niir', 'PAL', 'GERBER_625', 1),
    _c('niir_hue', 'PAL', 'GERBER_625', 2),
    # 819-line AM proto-SECAM (protosecam.py)
    _c('protosecam', 'SECAM_1957', 'FRENCH_819', 1),
    _c('protosecam', 'SECAM_1957', 'FRENCH_819', 2, avg=True),
    # D2-MAC (mac.py)
    _c('mac', 'D2MAC_12MHZ', 'GERBER_625', 0),
    _c('mac', 'D2MAC_12MHZ', 'GERBER_625', 1, avg=True),
    _c('mac', 'D2MAC_7MHZ', 'GERBER_625', 3),
    # 1920-wide (36 MHz / 47 MHz sampling)
    _c('secam', 'SECAM_E', 'FRENCH_819', 1, width=1920),
    _c('pal_d', 'PAL', 'GERBER_625', 2, width=1920),
    _c('ntsc_3d', 'NTSC', 'NTSC_525', 1, width=1920),
    _c('mac', 'D2MAC_7MHZ', 'GERBER_625', 1, width=1920),
    _c('niir_hue', 'PAL', 'GERBER_625', 3, width=1920),
    # luma notch of the comb decoders (non-default knob notch=Q, comb.py:18-20,54-55,108-109, pal.py:227-228)
    _c('ntsc_comb', 'NTSC', 'NTSC_525', 3, notch=8.0),
    _c('ntsc_3d', 'NTSC', 'NTSC_525', 4, notch=4.0),
    _c('pal_d', 'PAL', 'GERBER_625', 4, notch=8.0),
    _c('pal_3d', 'PAL', 'GERBER_625', 5, notch=2.0, content='noise'),
    _c('pal_d', 'PAL', 'GERBER_625', 3, width=1920, notch=12.0),
    # other non-default knobs
    _c('pal_3d', 'PAL', 'GERBER_625', 4, opt='nosin'),
    _c('pal_3d', 'PAL', 'GERBER_625', 2, opt='nocos'),
    _c('pal_3d', 'PAL_M', 'NTSC_525', 1, opt='nocos', notch=6.0),
    _c('secam', 'SECAM', 'GERBER_625', 6, opt='altph'),
    _c('protosecam', 'SECAM_1957', 'FRENCH_819', 3, opt='noluma'),
    _c('ntsc_3d', 'NTSC', 'NTSC_525', 5, opt='minavg'),
    _c('ntsc_3d', 'NTSC443', 'NTSC_525', 6, opt='minavg', notch=5.0, content='noise'),
    _c('pal_3d', 'PAL', 'GERBER_625', 7, opt='minavg'),
    _c('pal_3d', 'PAL', 'GERBER_625', 0, opt='minavg', notch=3.0),
    # every preset / standard pair of BASELINE configs[4] at 1920 samples per line (23-47 MHz sampling: the multi-warp
    # kernels); the pairs not already covered above (SECAM_E, D2MAC_7MHZ, PAL, NTSC)
    _c('ntsc_3d', 'NTSC_A', 'BAIRD_405', 2, width=1920),
    _c('ntsc_3d', 'NTSC_I', 'GERBER_625', 3, width=1920),
    _c('ntsc_3d', 'NTSC_N', 'GERBER_625', 4, width=1920),
    _c('ntsc_3d', 'NTSC361', 'NTSC_525', 5, width=1920),
    _c('ntsc_3d', 'NTSC443', 'NTSC_525', 6, width=1920),
    _c('pal_d', 'PAL_M', 'NTSC_525', 1, width=1920),
    _c('pal_d', 'PAL_N', 'GERBER_625', 2, width=1920),
    _c('secam', 'SECAM_I', 'GERBER_625', 1, width=1920, avg=True),
    _c('secam', 'SECAM_II', 'GERBER_625', 2, width=1920, avg=True),
    _c('secam', 'SECAM_III', 'GERBER_625', 3, width=1920, avg=True),
    _c('secam', 'SECAM_A', 'BAIRD_405', 4, width=1920, avg=True),
    _c('secam', 'SECAM_M', 'NTSC_525', 5, width=1920, avg=True),
    _c('secam', 'SECAM_N', 'GERBER_625', 6, width=1920, avg=True),
    _c('protosecam', 'SECAM_1957', 'FRENCH_819', 2, width=1920, avg=True),
    # the fifth line standard (line.py:46)
    _c('pal_s', 'PAL', 'BELGIAN_819', 3),
    _c('ntsc_comb', 'NTSC443', 'BELGIAN_819', 4, width=1920),
    # SimpleCombModem / Simple3DCombModem over other backends (comb.py:71-127; cli.py:52 is the first one)
    _c('scomb+niir_hue', 'PAL', 'GERBER_625', 1),
    _c('scomb+niir', 'PAL', 'GERBER_625', 2, notch=4.0),
    _c('scomb3+niir', 'PAL', 'GERBER_625', 3),
    _c('scomb+pal_s', 'PAL', 'GERBER_625', 4, notch=6.0),
    _c('scomb3+pal_s', 'PAL', 'GERBER_625', 5),
    _c('scomb+ntsc', 'NTSC', 'NTSC_525', 6, opt='minavg'),
    _c('scomb3+ntsc', 'NTSC', 'NTSC_525', 7, opt='minavg', notch=5.0),
    _c('scomb+ntsc_comb', 'NTSC', 'NTSC_525', 1),
    _c('scomb3+pal_s', 'PAL_M', 'NTSC_525', 2, width=1920),
    # NtscCombModem where the line comb is unusable (custom subcarrier; ntsc.py:55-59,71-72), alone and under Simple3DCombModem
    _c('ntsc_comb', 'NTSC_NOCOMB', 'NTSC_525', 2),
    _c('ntsc_3d', 'NTSC_NOCOMB', 'NTSC_525', 3, notch=3.0),
    # BASELINE configs[0] and configs[1] at their own size: one whole frame each
    _c('ntsc', 'NTSC', 'NTSC_525', 0, height=480, seed=0),
    _c('pal_d', 'PAL', 'GERBER_625', 0, height=576, seed=0),
]

FLOAT_ROWS = (1, 10, 22)   # rows whose float64 composite / RGB lines are stored: field top, interior, field bottom

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
# The decoded frame `rgb_u8` of a whole-frame fixture does not compress below 1 MB, so it is stored in chunks of this many
# rows: the first chunk in <id>.npz with the other arrays, chunk k in <id>.part<k>.npz.
RGB_ROWS_PER_FILE = 192


def case_id(c):
    return '%s-%s-%dx%d-%s%s-f%d-%s%s' % (c.kind, c.variant, c.width, c.height, c.standard,
                                          '-avg' if c.chroma_avg else '', c.frame, c.content,
                                          ('-notch%g' % c.notch if c.notch else '') + ('-' + c.opt if c.opt else ''))


def save_golden(c, **arrays):
    base = os.path.join(GOLDEN_DIR, case_id(c))
    rgb = arrays.pop('rgb_u8')
    np.savez_compressed(base + '.npz', rgb_u8=rgb[:RGB_ROWS_PER_FILE], **arrays)
    for k, y in enumerate(range(RGB_ROWS_PER_FILE, rgb.shape[0], RGB_ROWS_PER_FILE), 1):
        np.savez_compressed('%s.part%d.npz' % (base, k), rgb_u8=rgb[y:y + RGB_ROWS_PER_FILE])
    return base + '.npz'


def load_golden(c):
    """The arrays of case c's fixture (comp_u8, rgb_u8, comp_f64, rgb_f64), the chunks of rgb_u8 joined."""
    base = os.path.join(GOLDEN_DIR, case_id(c))
    with np.load(base + '.npz') as f:
        g = dict(f)
    chunks, k = [g['rgb_u8']], 1
    while os.path.exists('%s.part%d.npz' % (base, k)):
        with np.load('%s.part%d.npz' % (base, k)) as f:
            chunks.append(f['rgb_u8'])
        k += 1
    g['rgb_u8'] = np.concatenate(chunks)
    return g


# BASELINE configs 1-5 at their full size (tests/test_oracle_vs_reference.py).  A whole frame does not fit a fixture, so
# full-<id>.npz holds the SHA-256 of each u8 frame (comp, rgb) with its shape, a few of its rows for diagnosis, and
# `source`: 'reference' where the frames are the reference's own output, 'oracle' where they pin the oracle's output
# until tests/golden/make_golden.py --full is run against the reference.
FULL_CASES = [
    Case('ntsc', 'NTSC', 720, 480, None, False, 0, 0, 'smooth'),          # BASELINE config 1
    Case('pal_d', 'PAL', 720, 576, None, False, 0, 0, 'smooth'),          # BASELINE config 2
    Case('ntsc_3d', 'NTSC', 720, 480, None, False, 599, 3, 'smooth'),     # BASELINE config 3 (last frame)
    Case('secam', 'SECAM', 720, 576, None, True, 7, 4, 'noise'),          # BASELINE config 4a
    Case('niir_hue', 'PAL', 720, 576, None, False, 999, 5, 'smooth'),     # BASELINE config 4b
    Case('mac', 'D2MAC_7MHZ', 1920, 1080, 'GERBER_625', False, 2, 6, 'smooth'),   # BASELINE config 5 sample
]
FULL_SAMPLE_ROWS = 8


def frame_digest(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def save_full(c, comp_u8, rgb_u8, source):
    rows = np.linspace(0, comp_u8.shape[0] - 1, FULL_SAMPLE_ROWS).round().astype(np.int64)
    path = os.path.join(GOLDEN_DIR, 'full-%s.npz' % case_id(c))
    np.savez_compressed(path, source=np.array(source), rows=rows,
                        comp_sha256=frame_digest(comp_u8), comp_shape=np.array(comp_u8.shape), comp_rows=comp_u8[rows],
                        rgb_sha256=frame_digest(rgb_u8), rgb_shape=np.array(rgb_u8.shape), rgb_rows=rgb_u8[rows])
    return path


def load_full(c):
    with np.load(os.path.join(GOLDEN_DIR, 'full-%s.npz' % case_id(c))) as f:
        return dict(f)
