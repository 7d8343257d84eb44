#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the UNMODIFIED reference, a checkout of kFYatek/color_modem.

    COLOR_MODEM_REFERENCE=<checkout> python tests/golden/make_golden.py [--missing]
                                                          (--missing: only the cases without a fixture yet)
    [COLOR_MODEM_REFERENCE=<checkout>] python tests/golden/make_golden.py --full

For every case in tests/cases.py this imports kFYatek/color_modem read-only, installs the scipy
``iirdesign`` validation shim of SURVEY.md §8c (needed by NTSC / PAL-M / PAL-N presets on scipy >= 1.6,
bit-identical to stock scipy on valid input), builds the reference modem composition and calls the
reference's own frame driver ``ImageModem.modulate`` / ``.demodulate`` (image.py:27,58).  Stored per case:

    comp_u8   [H, Wc]     composite frame as produced by ImageModem.modulate
    rgb_u8    [H, Wo, 3]  frame decoded by ImageModem.demodulate from comp_u8
    comp_f64  [R, Wc]     float64 level-mapped composite (argument of image._as_bytes) for rows FLOAT_ROWS
    rgb_f64   [R, Wo, 3]  float64 decoded RGB (arguments of image._as_bytes) for rows FLOAT_ROWS

The inputs are regenerated from color_modem_b200.synth (integer-only, platform independent).  rgb_u8 of a whole
frame is split over <id>.npz and <id>.part<k>.npz (tests/cases.py: save_golden / load_golden).

--full writes the digests of the whole frames of FULL_CASES (full-<id>.npz): from the reference when
COLOR_MODEM_REFERENCE is set; without it from a whole-frame fixture of the same frame generated from the
reference, checked against the oracle; else from the oracle, marked source 'oracle'.
"""
import os
import sys
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.dont_write_bytecode = True
os.environ['PYTHONDONTWRITEBYTECODE'] = '1'

import numpy as np                                             # noqa: E402

from refload import load_reference, reference_available       # noqa: E402
from cases import GOLDEN_CASES, FLOAT_ROWS, FULL_CASES, case_id, load_golden, save_full, save_golden   # noqa: E402
from color_modem_b200.synth import synth_frames_u8             # noqa: E402


def make_full():
    import oracle
    from oracle import frame as oframe
    from PIL import Image
    ref = load_reference() if reference_available() else None
    for c in FULL_CASES:
        rgb = synth_frames_u8(1, c.height, c.width, first_frame=c.frame, seed=c.seed, kind=c.content)[0]
        if ref is not None:
            driver = ref.image.ImageModem(ref.make_modem(c))
            comp_img = driver.modulate(Image.fromarray(rgb, 'RGB'), c.frame)
            comp, out, source = np.asarray(comp_img), np.asarray(driver.demodulate(comp_img, c.frame)), 'reference'
        else:
            om = oracle.build(oracle.ModemSpec(c.kind, c.variant, c.width, c.height, c.standard, c.chroma_avg, c.notch,
                                               c.opt))
            comp = oframe.encode_frame_u8(om, c.frame, rgb)
            out = oframe.decode_frame_u8(om, c.frame, comp)
            source = 'oracle'
            same = [g for g in GOLDEN_CASES if g._replace(standard=c.standard) == c]
            if same:
                g = load_golden(same[0])
                assert np.array_equal(comp, g['comp_u8']) and np.array_equal(out, g['rgb_u8']), case_id(c)
                source = 'reference'
        print('%-50s %s  %s' % (case_id(c), source, save_full(c, comp, out, source)))


def main():
    warnings.filterwarnings('ignore')
    if '--full' in sys.argv:
        return make_full()
    ref = load_reference()
    from PIL import Image
    only_missing = '--missing' in sys.argv
    for c in GOLDEN_CASES:
        if only_missing and os.path.exists(os.path.join(HERE, case_id(c) + '.npz')):
            continue
        rgb = synth_frames_u8(1, c.height, c.width, first_frame=c.frame, seed=c.seed, kind=c.content)[0]
        modem = ref.make_modem(c)
        driver = ref.image.ImageModem(modem)
        with ref.capture_floats() as cap:
            comp_img = driver.modulate(Image.fromarray(rgb, 'RGB'), c.frame)
        comp = np.asarray(comp_img)
        comp_f = ref.rows_in_raster_order(cap, c.height, 1)
        with ref.capture_floats() as cap:
            out_img = driver.demodulate(comp_img, c.frame)
        out = np.asarray(out_img)
        rgb_f = ref.rows_in_raster_order(cap, c.height, 3)
        rows = [r for r in FLOAT_ROWS if r < c.height]
        path = save_golden(c, comp_u8=comp, rgb_u8=out,
                           comp_f64=comp_f[rows, 0], rgb_f64=np.moveaxis(rgb_f[rows], 1, -1))
        print('%-60s comp %s rgb %s  %d KB' % (case_id(c), comp.shape, out.shape, os.path.getsize(path) // 1024))


if __name__ == '__main__':
    main()
