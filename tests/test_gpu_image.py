"""GPU: the literal drop-in calls of the reference's frame driver — ``ImageModem(modem).modulate(img, frame)`` and
``.demodulate(img, frame)`` with PIL images (image.py:27-84) — against the bytes the reference itself produced
(tests/golden/*.npz), including the automatic mode conversion of image.py:28-29,60-61 and the integer-width form of
``MacModem`` (mac.py:18-21)."""
import numpy as np
import pytest

from cases import GOLDEN_CASES, case_id, load_golden
from product import make_modem
from color_modem_b200.image import ImageModem
from color_modem_b200.synth import synth_frames_u8

pytestmark = pytest.mark.gpu

PICK = {('pal_d', 'PAL', 720, 24, ''), ('ntsc_3d', 'NTSC', 720, 24, ''), ('secam', 'SECAM', 720, 24, ''),
        ('mac', 'D2MAC_7MHZ', 720, 24, ''), ('pal_s', 'PAL', 720, 24, ''), ('ntsc', 'NTSC', 720, 480, ''),
        ('pal_d', 'PAL', 720, 576, '')}
_seen = set()
CASES = []
for _c in GOLDEN_CASES:
    _k = (_c.kind, _c.variant, _c.width, _c.height, _c.opt)
    if _k in PICK and not _c.notch and (_k, _c.standard) not in _seen and _c.content == 'smooth':
        _seen.add((_k, _c.standard))
        CASES.append(_c)


def _lsb(a, b):
    return int(np.abs(a.astype(np.int32) - b.astype(np.int32)).max())


@pytest.mark.parametrize('c', CASES, ids=case_id)
def test_pil_images_against_reference_bytes(c, cuda_required):
    from PIL import Image
    g = load_golden(c)
    rgb = synth_frames_u8(1, c.height, c.width, first_frame=c.frame, seed=c.seed, kind=c.content)[0]
    driver = ImageModem(make_modem(c))
    comp_img = driver.modulate(Image.fromarray(rgb, 'RGB'), c.frame)
    assert comp_img.mode == 'L' and comp_img.size == (g['comp_u8'].shape[1], c.height)
    assert _lsb(np.asarray(comp_img), g['comp_u8']) <= 1
    out_img = driver.demodulate(Image.fromarray(g['comp_u8'], 'L'), c.frame)
    assert out_img.mode == 'RGB' and out_img.size == (g['rgb_u8'].shape[1], c.height)
    assert _lsb(np.asarray(out_img), g['rgb_u8']) <= 1


def test_mode_conversion_like_the_reference(cuda_required):
    """image.py:28-29 / 60-61: any other PIL mode is converted to 'RGB' / 'L' first."""
    from PIL import Image
    c = [x for x in CASES if x.kind == 'pal_d' and x.height == 24][0]
    g = load_golden(c)
    rgb = synth_frames_u8(1, c.height, c.width, first_frame=c.frame, seed=c.seed, kind=c.content)[0]
    driver = ImageModem(make_modem(c))
    img = Image.fromarray(rgb, 'RGB')
    direct = np.asarray(driver.modulate(img, c.frame))
    # RGBA and a palette image that round-trips losslessly to the same RGB pixels
    assert np.array_equal(np.asarray(driver.modulate(img.convert('RGBA'), c.frame)), direct)
    pal_img = img.convert('P', palette=Image.ADAPTIVE, colors=256)
    want = np.asarray(driver.modulate(pal_img.convert('RGB'), c.frame))
    assert np.array_equal(np.asarray(driver.modulate(pal_img, c.frame)), want)
    # composite handed over as RGB: converted to 'L' (ITU-R 601 luma of three equal channels = the value itself)
    comp = Image.fromarray(g['comp_u8'], 'L')
    out = np.asarray(driver.demodulate(comp, c.frame))
    assert np.array_equal(np.asarray(driver.demodulate(comp.convert('RGB'), c.frame)), out)
    assert _lsb(out, g['rgb_u8']) <= 1


def test_mac_integer_width(cuda_required):
    """MacModem(line_config, 720) is MacModem(line_config, MacVariant.D2MAC_7MHZ) (mac.py:18-21)."""
    import torch
    from color_modem_b200.color import mac
    from color_modem_b200.line import LineConfig, LineStandard
    lc = LineConfig((720, 24), LineStandard.GERBER_625)
    a, b = mac.MacModem(lc, 720), mac.MacModem(lc, mac.MacVariant.D2MAC_7MHZ)
    rgb = torch.from_numpy(synth_frames_u8(2, 24, 720, seed=3)).cuda()
    ca, cb = a.encode_frames(rgb), b.encode_frames(rgb)
    assert torch.equal(ca, cb)
    assert torch.equal(a.decode_frames(ca), b.decode_frames(cb))
    assert mac.MacModem(lc, 540).composite_width == 540
