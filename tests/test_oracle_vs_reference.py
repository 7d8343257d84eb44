"""CPU: the oracle at full frame size (BASELINE configs 1-5) against the stored frames of tests/golden/full-*.npz, byte for
byte; where COLOR_MODEM_REFERENCE names a checkout of the reference (tests/refload.py), also against the live reference."""
import warnings

import numpy as np
import pytest

import oracle
from oracle import frame as oframe
from cases import FULL_CASES, frame_digest, load_full
from refload import reference_available, load_reference
from color_modem_b200.synth import synth_frames_u8


def _assert_stored(frame, g, name):
    assert frame.shape == tuple(g[name + '_shape'])
    diff = np.nonzero((frame[g['rows']] != g[name + '_rows']).reshape(len(g['rows']), -1).any(axis=1))[0]
    assert not len(diff), '%s differs from the %s frame on rows %s' % (name, g['source'], g['rows'][diff])
    assert np.array_equal(frame_digest(frame), g[name + '_sha256']), '%s differs from the %s frame' % (name, g['source'])


@pytest.mark.parametrize('c', FULL_CASES, ids=lambda c: '%s-%s-%dx%d' % (c.kind, c.variant, c.width, c.height))
def test_full_frame_u8_identical(c):
    rgb = synth_frames_u8(1, c.height, c.width, first_frame=c.frame, seed=c.seed, kind=c.content)[0]
    modem = oracle.build(oracle.ModemSpec(c.kind, c.variant, c.width, c.height, c.standard, c.chroma_avg, c.notch, c.opt))
    comp = oframe.encode_frame_u8(modem, c.frame, rgb)
    g = load_full(c)
    _assert_stored(comp, g, 'comp')
    out = oframe.decode_frame_u8(modem, c.frame, comp)
    _assert_stored(out, g, 'rgb')
    if reference_available():
        warnings.filterwarnings('ignore')
        from PIL import Image
        ref = load_reference()
        driver = ref.image.ImageModem(ref.make_modem(c))
        comp_img = driver.modulate(Image.fromarray(rgb, 'RGB'), c.frame)
        assert np.array_equal(comp, np.asarray(comp_img))
        assert np.array_equal(out, np.asarray(driver.demodulate(comp_img, c.frame)))
