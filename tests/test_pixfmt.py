"""Planar YUV 4:2:0 picture format (color_modem_b200/pixfmt.py, cm_pixfmt.cu, the *_host_fmt calls, Y4M ingest, the CLI).

CPU: the numpy restatement of the integer conversion (oracle/yuv.py) against known values and its own rules, frame sizes,
Y4M headers and frame prefixes, command-line parsing.  GPU: both conversion kernels byte-identical to the restatement; the
yuv420p host pipelines, the composed wrapper and the command line equal the rgb24 paths with the device conversions around
them; the conversions can be captured in a CUDA graph."""
import os
import types

import numpy as np
import pytest

from color_modem_b200 import ingest
from color_modem_b200.__main__ import build_modem, main, parse
from color_modem_b200.pixfmt import PixelFormat, frame_bytes
from oracle import yuv as oy

SETS = [(m, r) for m in ('bt601', 'bt709') for r in ('limited', 'full')]


def _yuv_frame(w, h, y, u, v):
    f = np.empty((1, oy.frame_bytes(w, h)), np.uint8)
    py, pu, pv = oy.split_planes(f, w, h)
    py[...], pu[...], pv[...] = y, u, v
    return f


# ---- CPU ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('matrix,rng', SETS)
def test_oracle_black_white_grey(matrix, rng):
    lo, hi = (16, 235) if rng == 'limited' else (0, 255)
    for yv, want in ((lo, 0), (hi, 255)):
        rgb = oy.yuv420p_to_rgb(_yuv_frame(8, 3, yv, 128, 128), 8, 3, matrix, rng)
        assert (rgb == want).all(), (matrix, rng, yv)
    grey = np.repeat(np.arange(256, dtype=np.uint8), 3).reshape(1, 16, 16, 3)
    _, u, v = oy.split_planes(oy.rgb_to_yuv420p(grey, matrix, rng), 16, 16)
    assert (u == 128).all() and (v == 128).all()


def _bars(matrix, rng):
    """75 % colour bars: the textbook float definition, rounded."""
    kr, kb = oy.MATRICES[matrix]
    out = []
    for r, g, b in ((1, 1, 1), (1, 1, 0), (0, 1, 1), (0, 1, 0), (1, 0, 1), (1, 0, 0), (0, 0, 1)):
        r, g, b = 0.75 * r, 0.75 * g, 0.75 * b
        ey = kr * r + (1 - kr - kb) * g + kb * b
        ecb, ecr = (b - ey) / (2 * (1 - kb)), (r - ey) / (2 * (1 - kr))
        if rng == 'limited':
            out.append((16 + 219 * ey, 128 + 224 * ecb, 128 + 224 * ecr))
        else:
            out.append((255 * ey, 128 + 255 * ecb, 128 + 255 * ecr))
    return np.round(np.array(out))


# the printed 75 % bar tables (white, yellow, cyan, green, magenta, red, blue) of the two studio standards
TEXTBOOK_LIMITED = {
    'bt601': [(180, 128, 128), (162, 44, 142), (131, 156, 44), (112, 72, 58), (84, 184, 198), (65, 100, 212), (35, 212, 114)],
    'bt709': [(180, 128, 128), (168, 44, 136), (145, 147, 44), (133, 63, 52), (63, 193, 204), (51, 109, 212), (28, 212, 120)],
}


@pytest.mark.parametrize('matrix,rng', SETS)
def test_oracle_colour_bars(matrix, rng):
    rgb = np.zeros((1, 2, 14, 3), np.uint8)
    cols = [(1, 1, 1), (1, 1, 0), (0, 1, 1), (0, 1, 0), (1, 0, 1), (1, 0, 0), (0, 0, 1)]
    for i, c in enumerate(cols):
        rgb[0, :, 2 * i:2 * i + 2] = np.array(c) * 191
    y, u, v = oy.split_planes(oy.rgb_to_yuv420p(rgb, matrix, rng), 14, 2)
    got = np.stack([y[0, 0, 0::2], u[0, 0], v[0, 0]], axis=-1).astype(int)
    assert np.abs(got - _bars(matrix, rng)).max() <= 1, got
    if rng == 'limited':
        assert np.abs(got - np.array(TEXTBOOK_LIMITED[matrix])).max() <= 1, got
    back = oy.yuv420p_to_rgb(oy.rgb_to_yuv420p(rgb, matrix, rng), 14, 2, matrix, rng).astype(int)
    assert np.abs(back - rgb).max() <= 2


@pytest.mark.parametrize('matrix,rng', SETS)
def test_oracle_coefficient_rows(matrix, rng):
    c = oy.coefficients(matrix, rng)
    s = 219.0 / 255.0 if rng == 'limited' else 1.0
    assert c['YR'] + c['YG'] + c['YB'] == oy.round_half_away(65536 * s)
    assert c['UR'] + c['UG'] + c['UB'] == 0 and c['VR'] + c['VG'] + c['VB'] == 0
    worst = 255 * (abs(c['Y']) + abs(c['RV']) + abs(c['GU']) + abs(c['GV']) + abs(c['BU'])) + 4 * 255 * (
        abs(c['UR']) + abs(c['UG']) + abs(c['UB'])) + (1 << 26)
    assert worst < 2 ** 31                       # every intermediate fits in int32


def test_oracle_odd_height_and_rounding_by_hand():
    """The vectorised restatement against a per-pixel loop written from the rule, odd height included."""
    rng = np.random.default_rng(1)
    w, h = 8, 5
    rgb = rng.integers(0, 256, (1, h, w, 3), dtype=np.uint8)
    c = oy.coefficients('bt709', 'full')
    got = oy.rgb_to_yuv420p(rgb, 'bt709', 'full')
    gy, gu, gv = oy.split_planes(got, w, h)
    px = rgb[0].astype(int)
    for yy in range(h):
        for xx in range(w):
            r, g, b = px[yy, xx]
            assert gy[0, yy, xx] == min(255, max(0, (c['YR'] * r + c['YG'] * g + c['YB'] * b + 32768) >> 16))
    for cy in range((h + 1) // 2):
        for cx in range(w // 2):
            rows = [2 * cy, min(2 * cy + 1, h - 1)]
            su = sum(c['UR'] * px[r_, x_, 0] + c['UG'] * px[r_, x_, 1] + c['UB'] * px[r_, x_, 2]
                     for r_ in rows for x_ in (2 * cx, 2 * cx + 1))
            assert gu[0, cy, cx] == min(255, max(0, (su + 128 * (1 << 18) + (1 << 17)) >> 18))
    back = oy.yuv420p_to_rgb(got, w, h, 'bt709', 'full')
    yv = int(gy[0, 4, 6])
    uv, vv = int(gu[0, 2, 3]) - 128, int(gv[0, 2, 3]) - 128
    assert back[0, 4, 6, 0] == min(255, max(0, (c['Y'] * yv + c['RV'] * vv + 32768) >> 16))
    assert back[0, 4, 6, 1] == min(255, max(0, (c['Y'] * yv + c['GU'] * uv + c['GV'] * vv + 32768) >> 16))


def test_frame_bytes_and_format_checks():
    assert frame_bytes('yuv420p', 720, 576) == 720 * 576 * 3 // 2
    for w, h in ((720, 3), (724, 5), (1920, 7)):
        assert frame_bytes(PixelFormat('yuv420p'), w, h) == w * h + 2 * (w // 2) * ((h + 1) // 2) == oy.frame_bytes(w, h)
    assert frame_bytes(None, 720, 5) == frame_bytes('rgb24', 720, 5) == 720 * 5 * 3
    for bad in (dict(name='nv12'), dict(name='yuv420p', matrix='bt2020'), dict(name='yuv420p', range='tv')):
        with pytest.raises(ValueError):
            PixelFormat(**bad)
    assert PixelFormat('yuv420p', 'bt709', 'full').c_struct().matrix == 1


def _y4m(tmp_path, name, header, frames, frame_header=b'FRAME\n'):
    p = str(tmp_path / name)
    with open(p, 'wb') as f:
        f.write(header)
        for fr in frames:
            f.write(frame_header)
            f.write(fr.tobytes())
    return p


def test_y4m_header_and_frames(tmp_path):
    w, h, n = 16, 5, 4
    fb = oy.frame_bytes(w, h)
    frames = np.random.default_rng(2).integers(0, 256, (n, fb), dtype=np.uint8)
    hdr = b'YUV4MPEG2 W16 H5 F25:1 Ip A1:1 C420mpeg2 XYSCSS=420MPEG2 XCOLORRANGE=FULL\n'
    p = _y4m(tmp_path, 'a.y4m', hdr, frames)
    assert ingest.read_y4m_header(p) == hdr
    info = ingest.parse_y4m_header(hdr)
    assert (info['width'], info['height'], info['chroma'], info['range']) == (16, 5, '420mpeg2', 'full')
    assert ingest.parse_y4m_header(b'YUV4MPEG2 W8 H2 F25:1\n')['chroma'] == '420jpeg'         # no C tag: 4:2:0 jpeg
    assert ingest.parse_y4m_header(b'YUV4MPEG2 W8 H2 XCOLORRANGE=LIMITED\n')['range'] == 'limited'
    assert ingest.picture_format(p, PixelFormat('yuv420p', 'bt709', 'limited')) == PixelFormat('yuv420p', 'bt709', 'full')
    modem = types.SimpleNamespace(width=w, height=h, composite_width=w)
    src = ingest.open_source(modem, 'transcode', p, PixelFormat('yuv420p'))
    assert src.nframes == n
    buf = np.empty((3, fb), np.uint8)
    assert src.read_into(1, buf) == 3 and np.array_equal(buf, frames[1:])
    src.close()
    # write round trip: header written once, frames at their offsets, each behind FRAME\n
    out = str(tmp_path / 'o.y4m')
    hdr2 = ingest.y4m_with_width(hdr, 12)
    assert hdr2 == b'YUV4MPEG2 W12 H5 F25:1 Ip A1:1 C420mpeg2 XYSCSS=420MPEG2 XCOLORRANGE=FULL\n'
    dst = ingest.RawVideo(out, (fb,), 'a', header=len(hdr), prefix=ingest.Y4M_FRAME)
    dst.write_header(hdr)
    dst.write_at(2, frames[2:])
    dst.write_at(0, frames[:2])
    dst.close()
    assert open(out, 'rb').read() == open(p, 'rb').read()
    fresh = ingest.y4m_header(720, 576, 25.0, PixelFormat('yuv420p', range='full'))
    assert ingest.parse_y4m_header(fresh)['range'] == 'full' and b' F25:1 ' in fresh
    assert b' F30000:1001 ' in ingest.y4m_header(720, 480, 30000 / 1001, PixelFormat('yuv420p'))


def test_y4m_refusals(tmp_path):
    for tag in (b'C422', b'C444', b'Cmono', b'C420p10', b'C411'):
        with pytest.raises(ValueError, match='4:2:0'):
            ingest.parse_y4m_header(b'YUV4MPEG2 W16 H4 F25:1 ' + tag + b'\n')
    with pytest.raises(ValueError):
        ingest.parse_y4m_header(b'YUV4MPEG2 W16 F25:1\n')
    with pytest.raises(ValueError):
        ingest.parse_y4m_header(b'YUV4MPEG2 W16 H4 XCOLORRANGE=STUDIO\n')
    bad = str(tmp_path / 'bad.png.y4m')
    with open(bad, 'wb') as f:
        f.write(b'\x89PNG\r\n')
    with pytest.raises(ValueError):
        ingest.read_y4m_header(bad)
    w, h = 16, 4
    frames = np.zeros((2, oy.frame_bytes(w, h)), np.uint8)
    p = _y4m(tmp_path, 'params.y4m', b'YUV4MPEG2 W16 H4 F25:1\n', frames, frame_header=b'FRAME Ixx\n')
    src = ingest.open_source(types.SimpleNamespace(width=w, height=h, composite_width=w), 'modulate', p, PixelFormat('yuv420p'))
    with pytest.raises(ValueError, match='FRAME'):
        src.read_into(0, np.empty((2, oy.frame_bytes(w, h)), np.uint8))
    src.close()


def test_cli_pixel_format_flags(tmp_path):
    a = parse(['transcode', '--modem', 'pal-d', '--size', '720x576', 'in.yuv', 'out.yuv'])
    assert a.raw and a.pix_fmt == PixelFormat('yuv420p', 'bt601', 'limited')
    a = parse(['modulate', '--modem', 'pal-d', '--size', '720x576', '--matrix', 'bt709', '--range', 'full', 'in.yuv', 'c.gray'])
    assert a.pix_fmt == PixelFormat('yuv420p', 'bt709', 'full')
    a = parse(['demodulate', '--modem', 'pal-d', '--size', '720x576', 'c.gray', 'out.y4m'])
    assert a.pix_fmt.name == 'yuv420p'
    a = parse(['transcode', '--modem', 'pal-d', '--size', '720x576', '--pix-fmt', 'yuv420p', 'in.raw', 'out.raw'])
    assert a.pix_fmt.name == 'yuv420p'
    a = parse(['transcode', '--modem', 'pal-d', '--size', '720x576', 'in.rgb', 'out.rgb'])
    assert a.pix_fmt == PixelFormat('rgb24')
    p = _y4m(tmp_path, 'in.y4m', b'YUV4MPEG2 W720 H24 F25:1 C420jpeg\n', np.zeros((1, oy.frame_bytes(720, 24)), np.uint8))
    a = parse(['transcode', '--modem', 'pal-d', p, 'out.y4m'])
    assert a.size == (720, 24) and a.pix_fmt.name == 'yuv420p'
    for argv in (['transcode', '--modem', 'pal-d', 'in.yuv', 'out.yuv'],                         # raw .yuv needs --size
                 ['transcode', '--modem', 'pal-d', '--size', '720x576', '--pix-fmt', 'rgb24', 'in.yuv', 'out.yuv'],
                 ['transcode', '--modem', 'pal-d', '--size', '720x576', '--range', 'tv', 'in.yuv', 'out.yuv'],
                 ['transcode', '--modem', 'pal-d', str(tmp_path / 'missing.y4m'), 'out.y4m']):
        with pytest.raises(SystemExit):
            parse(argv)


# ---- GPU ----------------------------------------------------------------------------------------------------------
def _pf(matrix, rng):
    return PixelFormat('yuv420p', matrix, rng)


@pytest.mark.gpu
@pytest.mark.parametrize('n', [1, 70])
@pytest.mark.parametrize('h', [3, 5, 576])
@pytest.mark.parametrize('w', [720, 724, 1920])
def test_conversion_kernels_match_the_oracle(w, h, n, cuda_required):
    """Random bytes (every value, Y' outside 16..235, chroma extremes that clip): both kernels byte for byte; three frames of
    the batch are checked (the frame index is the grid's z)."""
    import torch
    from color_modem_b200.pixfmt import from_rgb24, to_rgb24
    g = torch.Generator(device='cuda').manual_seed(w * 1000 + h * 10 + n)
    fb = frame_bytes('yuv420p', w, h)
    yuv = torch.randint(0, 256, (n, fb), dtype=torch.uint8, device='cuda', generator=g)
    rgb = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, device='cuda', generator=g)
    pick = sorted({0, n // 2, n - 1})
    y_np, r_np = yuv[pick].cpu().numpy(), rgb[pick].cpu().numpy()
    for matrix, rng in SETS:
        fmt = _pf(matrix, rng)
        got_rgb = to_rgb24(yuv, fmt, w, h)
        got_yuv = from_rgb24(rgb, fmt)
        torch.cuda.synchronize()
        assert np.array_equal(got_rgb[pick].cpu().numpy(), oy.yuv420p_to_rgb(y_np, w, h, matrix, rng)), (matrix, rng)
        assert np.array_equal(got_yuv[pick].cpu().numpy(), oy.rgb_to_yuv420p(r_np, matrix, rng)), (matrix, rng)


@pytest.mark.gpu
def test_conversion_arguments_are_checked(cuda_required):
    import torch
    from color_modem_b200.pixfmt import to_rgb24
    from color_modem_b200 import _native as N
    import ctypes as C
    yuv = torch.zeros((1, frame_bytes('yuv420p', 720, 4)), dtype=torch.uint8, device='cuda')
    rgb = torch.zeros((1, 4, 720, 3), dtype=torch.uint8, device='cuda')
    lib = N.load()
    st = torch.cuda.current_stream().cuda_stream
    for f, w in ((N.PixFmt(1, 2, 0, 0), 720), (N.PixFmt(1, 0, 5, 0), 720), (N.PixFmt(0, 0, 0, 0), 720),
                 (N.PixFmt(1, 0, 0, 0), 718)):
        assert lib.cm_yuv420p_to_rgb24(C.byref(f), yuv.data_ptr(), rgb.data_ptr(), w, 4, 1, st) == -1
        assert lib.cm_rgb24_to_yuv420p(C.byref(f), rgb.data_ptr(), yuv.data_ptr(), w, 4, 1, st) == -1
    with pytest.raises(ValueError):
        to_rgb24(yuv, PixelFormat('rgb24'), 720, 4)
    m = build_modem('pal-d', (720, 24), None, 'GERBER_625')
    bad = N.PixFmt(1, 7, 0, 0)
    comp = np.zeros((1, 24, 720), np.uint8)
    pic = np.zeros((1, frame_bytes('yuv420p', 720, 24)), np.uint8)
    assert lib.cm_decode_frames_host_fmt(m._handle(), comp.ctypes.data, pic.ctypes.data, 0, 1, C.byref(bad)) == -1


MODEMS = [('pal-d', 'GERBER_625'), ('ntsc-3d', 'NTSC_525'), ('secam-avg', 'GERBER_625'), ('niir-hue', 'GERBER_625'),
          ('mac', 'GERBER_625'), ('niir-hue-comb', 'GERBER_625')]


@pytest.mark.gpu
@pytest.mark.parametrize('h', [24, 35])
@pytest.mark.parametrize('name,std', MODEMS)
def test_yuv_batches_equal_the_rgb_path(name, std, h, cuda_required):
    """transcode / modulate / demodulate with yuv420p = the rgb24 path between to_rgb24 and from_rgb24."""
    import torch
    from color_modem_b200.image import ImageModem
    from color_modem_b200.pixfmt import from_rgb24, to_rgb24
    w, n, first = 720, 2 if name.endswith('comb') else 5, 7
    fmt = _pf(*SETS[(len(name) + h) % 4])
    im = ImageModem(build_modem(name, (w, h), None, std))
    wo = im._modem.output_width
    assert wo == 720
    yuv = np.random.default_rng(h).integers(0, 256, (n, frame_bytes(fmt, w, h)), dtype=np.uint8)
    rgb = to_rgb24(torch.from_numpy(yuv).cuda(), fmt, w, h).cpu().numpy()

    def to_yuv(x):
        return from_rgb24(torch.from_numpy(x).cuda(), fmt).cpu().numpy()

    comp_ref, out_ref = im.transcode_batch(rgb, first)
    comp, out = im.transcode_batch(yuv, first, pix_fmt=fmt)
    assert out.shape == (n, frame_bytes(fmt, wo, h))
    assert np.array_equal(comp, comp_ref), name
    assert np.array_equal(out, to_yuv(out_ref)), name
    c2, o2 = im.transcode_batch(yuv, first, want_composite=False, pix_fmt=fmt)
    assert c2 is None and np.array_equal(o2, out)
    assert np.array_equal(im.modulate_batch(yuv, first, pix_fmt=fmt), im.modulate_batch(rgb, first)), name
    assert np.array_equal(im.demodulate_batch(comp_ref, first, pix_fmt=fmt), to_yuv(im.demodulate_batch(comp_ref, first)))


@pytest.mark.gpu
def test_yuv_bt709_hd(cuda_required):
    import torch
    from color_modem_b200.image import ImageModem
    from color_modem_b200.pixfmt import from_rgb24, to_rgb24
    from color_modem_b200.synth import synth_frames_u8
    w, h, n = 1920, 1080, 8
    fmt = _pf('bt709', 'limited')
    m = build_modem('pal-d', (w, h), 'PAL_N', 'GERBER_625')
    yuv = from_rgb24(torch.from_numpy(synth_frames_u8(n, h, w, seed=4)).cuda(), fmt)
    rgb = to_rgb24(yuv, fmt, w, h)
    ref = from_rgb24(m.decode_frames(m.encode_frames(rgb, first_frame=3), first_frame=3), fmt).cpu().numpy()
    _, out = ImageModem(m).transcode_batch(yuv.cpu().numpy(), 3, pix_fmt=fmt)
    assert np.array_equal(out, ref)


@pytest.mark.gpu
@pytest.mark.parametrize('n', [17, 33, 129])
def test_host_chunks_equal_one_device_call(n, cuda_required):
    """The host pipelines cut a batch into 32-frame chunks; the bytes equal one device-resident call on the whole batch."""
    import torch
    from color_modem_b200.pixfmt import from_rgb24, to_rgb24
    w, h = 720, 24
    fmt = _pf('bt601', 'full')
    m = build_modem('pal-d', (w, h), None, 'GERBER_625')
    yuv = np.random.default_rng(n).integers(0, 256, (n, frame_bytes(fmt, w, h)), dtype=np.uint8)
    comp_d = m.encode_frames(to_rgb24(torch.from_numpy(yuv).cuda(), fmt, w, h), first_frame=11)
    out_d = from_rgb24(m.decode_frames(comp_d, first_frame=11), fmt).cpu().numpy()
    comp_d = comp_d.cpu().numpy()
    comp, out = m.transcode_frames_host(yuv, 11, pix_fmt=fmt)
    assert np.array_equal(comp, comp_d) and np.array_equal(out, out_d)
    assert np.array_equal(m.encode_frames_host(yuv, 11, pix_fmt=fmt), comp_d)
    assert np.array_equal(m.decode_frames_host(comp_d, 11, pix_fmt=fmt), out_d)


@pytest.mark.gpu
def test_conversions_can_be_captured_in_a_cuda_graph(cuda_required):
    import torch
    from color_modem_b200 import _native as N
    from color_modem_b200.pixfmt import from_rgb24, to_rgb24
    w, h = 720, 64
    fmt = _pf('bt709', 'full')
    m = build_modem('pal-d', (w, h), None, 'GERBER_625')
    yuv = torch.from_numpy(np.random.default_rng(3).integers(0, 256, (1, frame_bytes(fmt, w, h)), dtype=np.uint8)).cuda()
    rgb = to_rgb24(yuv, fmt, w, h)
    comp = m.encode_frames(rgb)
    out = m.decode_frames(comp)
    res = from_rgb24(out, fmt)
    ref = res.clone()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        to_rgb24(yuv, fmt, w, h, out=rgb)
        m.encode_frames(rgb, out=comp)
        m.decode_frames(comp, out=out)
        from_rgb24(out, fmt, out=res)
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    launches = N.launch_count()
    with torch.cuda.graph(g, stream=s):
        to_rgb24(yuv, fmt, w, h, out=rgb)
        m.encode_frames(rgb, out=comp)
        m.decode_frames(comp, out=out)
        from_rgb24(out, fmt, out=res)
    assert N.launch_count() - launches >= 4            # the conversions count as launches
    res.zero_()
    rgb.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(res, ref)


@pytest.mark.gpu
@pytest.mark.parametrize('ext', ['.y4m', '.yuv'])
def test_cli_yuv_files_equal_the_batch_api(ext, tmp_path, cuda_required):
    w, h, n = 720, 32, 7
    fmt = _pf('bt601', 'full' if ext == '.y4m' else 'limited')
    fb = frame_bytes(fmt, w, h)
    yuv = np.random.default_rng(9).integers(0, 256, (n, fb), dtype=np.uint8)
    hdr = b'YUV4MPEG2 W720 H32 F25:1 Ip A1:1 C420paldv XCOLORRANGE=FULL\n'
    if ext == '.y4m':
        src = _y4m(tmp_path, 'in.y4m', hdr, yuv)
        size = []
    else:
        src = str(tmp_path / 'in.yuv')
        yuv.tofile(src)
        size = ['--size', '%dx%d' % (w, h)]

    def frames_of(path, count):
        data = np.fromfile(path, np.uint8)
        if ext == '.y4m':
            assert bytes(data[:len(hdr)]) == hdr
            rows = data[len(hdr):].reshape(count, 6 + fb)
            assert (rows[:, :6] == np.frombuffer(b'FRAME\n', np.uint8)).all()
            return rows[:, 6:]
        return data.reshape(count, fb)

    m = build_modem('pal-d', (w, h), None, 'GERBER_625')
    comp_ref, out_ref = m.transcode_frames_host(yuv, 0, pix_fmt=fmt)
    out, comp = str(tmp_path / ('out' + ext)), str(tmp_path / 'comp.gray')
    # --range full on the .yuv path; the Y4M header's XCOLORRANGE=FULL overrides the default limited
    rng_args = [] if ext == '.y4m' else ['--range', fmt.range]
    assert main(['transcode', '--modem', 'pal-d', '--standard', 'GERBER_625', '--batch', '3'] + size + rng_args +
                [src, out, comp]) == 0
    assert np.array_equal(np.fromfile(comp, np.uint8).reshape(n, h, w), comp_ref)
    assert np.array_equal(frames_of(out, n), out_ref)
    # --frames: absolute frame numbers are kept, the output starts at its first frame
    part = str(tmp_path / ('part' + ext))
    assert main(['transcode', '--modem', 'pal-d', '--standard', 'GERBER_625', '--frames', '2:5'] + size + rng_args +
                [src, part]) == 0
    assert np.array_equal(frames_of(part, 3), out_ref[2:5])
    # two frame ranges written into one file (what --devices does, one process per range)
    two = str(tmp_path / ('two' + ext))
    open(two, 'wb').close()
    for rng in ((3, n), (0, 3)):
        ingest.run_file(m, 'transcode', src, two, frames=rng, batch=2, out_offset=rng[0], pix_fmt=fmt)
    assert np.array_equal(frames_of(two, n), out_ref)
    # demodulate of the composite to the picture format
    dem = str(tmp_path / ('dem' + ext))
    open(dem, 'wb').close()
    ingest.run_file(m, 'demodulate', comp, dem, batch=4, pix_fmt=fmt)
    data = np.fromfile(dem, np.uint8)
    if ext == '.y4m':
        dh = ingest.read_y4m_header(dem)
        assert ingest.parse_y4m_header(dh)['range'] == 'full'
        data = data[len(dh):].reshape(n, 6 + fb)[:, 6:]
    assert np.array_equal(data.reshape(n, fb), out_ref)
    assert os.path.getsize(out) == os.path.getsize(two)
