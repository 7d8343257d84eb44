"""CPU: the oracle reproduces every golden fixture generated from the reference itself (tests/golden/make_golden.py)."""
import numpy as np
import pytest

import oracle
from oracle import frame as oframe
from cases import GOLDEN_CASES, FLOAT_ROWS, case_id, load_golden
from color_modem_b200.synth import synth_frames_u8


@pytest.mark.parametrize('c', GOLDEN_CASES, ids=case_id)
def test_oracle_matches_reference_golden(c):
    g = load_golden(c)
    modem = oracle.build(oracle.ModemSpec(c.kind, c.variant, c.width, c.height, c.standard, c.chroma_avg, c.notch, c.opt))
    rgb = synth_frames_u8(1, c.height, c.width, first_frame=c.frame, seed=c.seed, kind=c.content)[0]
    rows = list(FLOAT_ROWS)

    comp_f = oframe.composite_level(oframe.encode_frame_float(modem, c.frame, rgb))
    assert comp_f.shape == g['comp_u8'].shape
    np.testing.assert_allclose(comp_f[rows], g['comp_f64'], rtol=0, atol=1e-12)
    assert np.array_equal(oframe.to_u8(comp_f), g['comp_u8'])          # byte-exact composite frame

    rgb_f = oframe.decode_frame_float(modem, c.frame, g['comp_u8'])
    assert rgb_f.shape == g['rgb_u8'].shape
    np.testing.assert_allclose(rgb_f[rows], g['rgb_f64'], rtol=0, atol=1e-11)
    assert np.array_equal(oframe.to_u8(rgb_f), g['rgb_u8'])            # byte-exact decoded frame
