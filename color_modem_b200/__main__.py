"""Command line (SURVEY.md §8 f4; the reference's cli.py:18-65 with the composition chosen by name instead of by editing
the source).

    python -m color_modem_b200 OP --modem NAME [--variant V] [--standard S] [--size WxH] [--frames A:B]
                                  [--pix-fmt rgb24|yuv420p] [--matrix bt601|bt709] [--range limited|full]
                                  [--devices 0,1,...] [--batch N] INPUT OUTPUT [OUTPUT2]

OP       modulate | demodulate | transcode (modulate, then demodulate the result; OUTPUT2 = the composite)
INPUT    a picture (anything PIL opens; one frame, --size taken from it) or raw video: pictures (the input of modulate /
         transcode, the output of demodulate / transcode) as .rgb / .raw (rgb24 frames), .yuv (raw yuv420p frames) or .y4m
         (YUV4MPEG2, 8-bit 4:2:0; its header gives the size), the composite as .gray / .y (gray8, also for .raw input to
         demodulate).  --size is required for raw video other than .y4m input.
--pix-fmt picture format of the raw picture files: rgb24 (default) or yuv420p (implied by .yuv and .y4m).  yuv420p moves
         half the bytes of rgb24 over the host link; the conversion runs on the GPU.
--matrix / --range  colour matrix and quantisation range of yuv420p (default bt601, limited); a Y4M input's XCOLORRANGE
         overrides --range.  A Y4M output copies the Y4M input's header (W = the decoded width), or gets a fresh one.
--frames file frames [A, B) only; frame i of the file is absolute frame i
--devices comma-separated CUDA devices: the frame range is cut into one contiguous range per device, one process each
"""
import argparse
import os
import sys


def registry():
    """name -> (builder(line_config, variant_name or None), variant holder)"""
    from .color import ntsc, pal, secam, niir, protosecam, mac
    from . import comb

    def var(holder, name, default):
        return getattr(holder, name) if name else default

    NV, PV, SV = ntsc.NtscVariant, pal.PalVariant, secam.SecamVariant
    PSV, MV = protosecam.ProtoSecamVariant, mac.MacVariant
    return {
        'ntsc': lambda lc, v: ntsc.NtscModem(lc, var(NV, v, NV.NTSC)),
        'ntsc-comb': lambda lc, v: ntsc.NtscCombModem(lc, var(NV, v, NV.NTSC)),
        'ntsc-3d': lambda lc, v: comb.Simple3DCombModem(ntsc.NtscCombModem(lc, var(NV, v, NV.NTSC))),
        'pal-s': lambda lc, v: pal.PalSModem(lc, var(PV, v, PV.PAL)),
        'pal-d': lambda lc, v: pal.PalDModem(lc, var(PV, v, PV.PAL)),
        'pal-3d': lambda lc, v: pal.Pal3DModem(lc, var(PV, v, PV.PAL)),
        'secam': lambda lc, v: secam.SecamModem(lc, var(SV, v, SV.SECAM)),
        'secam-avg': lambda lc, v: comb.ColorAveragingModem(secam.SecamModem(lc, var(SV, v, SV.SECAM))),
        'niir': lambda lc, v: niir.NiirModem(lc, var(PV, v, PV.PAL)),
        'niir-hue': lambda lc, v: niir.HueCorrectingNiirModem(lc, var(PV, v, PV.PAL)),
        'niir-hue-comb': lambda lc, v: comb.SimpleCombModem(niir.HueCorrectingNiirModem(lc, var(PV, v, PV.PAL))),
        'protosecam': lambda lc, v: protosecam.ProtoSecamModem(lc, var(PSV, v, PSV.SECAM_1957)),
        'protosecam-avg': lambda lc, v: comb.ColorAveragingModem(protosecam.ProtoSecamModem(lc, var(PSV, v, PSV.SECAM_1957))),
        'mac': lambda lc, v: mac.MacModem(lc, var(MV, v, MV.D2MAC_12MHZ)),
        'mac-avg': lambda lc, v: comb.ColorAveragingModem(mac.MacModem(lc, var(MV, v, MV.D2MAC_12MHZ))),
    }


def build_modem(name, size, variant=None, standard=None):
    from .line import LineConfig, LineStandard
    std = getattr(LineStandard, standard) if standard else None
    reg = registry()
    if name not in reg:
        raise SystemExit('unknown --modem %r; one of: %s' % (name, ', '.join(sorted(reg))))
    return reg[name](LineConfig(tuple(size), std), variant)


def parse(argv=None):
    ap = argparse.ArgumentParser(prog='python -m color_modem_b200', description=__doc__.split('\n')[0])
    ap.add_argument('op', choices=['modulate', 'demodulate', 'transcode'])
    ap.add_argument('--modem', required=True)
    ap.add_argument('--variant', default=None)
    ap.add_argument('--standard', default=None, help='LineStandard name (default: detected from the height, line.py:34-46)')
    ap.add_argument('--size', default=None, help='WxH (raw video)')
    ap.add_argument('--frames', default=None, help='A:B, file frames [A, B)')
    ap.add_argument('--devices', default='0')
    ap.add_argument('--batch', type=int, default=64)
    ap.add_argument('--pix-fmt', default=None, choices=['rgb24', 'yuv420p'],
                    help='picture format of raw video (default rgb24; yuv420p implied by .yuv / .y4m)')
    ap.add_argument('--matrix', default='bt601', choices=['bt601', 'bt709'], help='yuv420p colour matrix')
    ap.add_argument('--range', default='limited', choices=['limited', 'full'],
                    help='yuv420p range (a Y4M input\'s XCOLORRANGE overrides it)')
    ap.add_argument('input')
    ap.add_argument('output')
    ap.add_argument('output2', nargs='?', default=None)
    a = ap.parse_args(argv)
    a.size = tuple(int(v) for v in a.size.lower().split('x')) if a.size else None
    if a.frames:
        lo, _, hi = a.frames.partition(':')
        a.frames = (int(lo or 0), int(hi) if hi else 1 << 62)
    a.devices = [int(d) for d in a.devices.split(',') if d != '']
    from . import ingest
    from .pixfmt import PixelFormat
    a.raw = os.path.splitext(a.input)[1].lower() in ('.rgb', '.raw', '.gray', '.y', '.yuv', '.y4m')
    implied = any(ingest.is_yuv(p) for p in ingest.picture_paths(a.op, a.input, a.output))
    if implied and a.pix_fmt == 'rgb24':
        ap.error('.yuv / .y4m files hold yuv420p frames, not --pix-fmt rgb24')
    a.pix_fmt = PixelFormat(a.pix_fmt or ('yuv420p' if implied else 'rgb24'), a.matrix, a.range)
    if a.raw and not a.size and a.op != 'demodulate' and ingest.is_y4m(a.input):
        try:
            info = ingest.parse_y4m_header(ingest.read_y4m_header(a.input))
        except (OSError, ValueError) as e:
            ap.error(str(e))
        a.size = (info['width'], info['height'])
    if a.raw and not a.size:
        ap.error('--size WxH is required for raw video')
    return a


def _worker(a, dev, frames, base):
    """One device, file frames [frames[0], frames[1]); output frame 0 is file frame `base`."""
    import torch
    from . import ingest
    torch.cuda.set_device(dev)
    modem = build_modem(a.modem, a.size, a.variant, a.standard)
    return ingest.run_file(modem, a.op, a.input, a.output, a.output2, frames=frames, batch=a.batch,
                           out_offset=frames[0] - base, pix_fmt=a.pix_fmt)


def main(argv=None):
    a = parse(argv)
    if not a.raw:                                           # one picture, exactly the reference's cli.py:18-65
        from PIL import Image
        from .image import ImageModem
        img = Image.open(a.input)
        modem = build_modem(a.modem, img.size, a.variant, a.standard)
        im = ImageModem(modem)
        frame = a.frames[0] if a.frames else 0
        if a.op == 'modulate':
            im.modulate(img, frame).save(a.output)
        elif a.op == 'demodulate':
            im.demodulate(img, frame).save(a.output)
        else:
            comp = im.modulate(img, frame)
            if a.output2:
                comp.save(a.output2)
            im.demodulate(comp, frame).save(a.output)
        return 0
    from . import ingest
    from .shard import frame_range
    probe = build_modem(a.modem, a.size, a.variant, a.standard)
    src = ingest.open_source(probe, a.op, a.input, a.pix_fmt)
    total = src.nframes
    src.close()
    lo, hi = a.frames if a.frames else (0, total)
    hi = min(hi, total)
    for path in (a.output, a.output2):                      # the workers write at frame offsets of existing files
        if path:
            open(path, 'wb').close()
    header = ingest.output_header(probe, a.op, a.input, a.output,
                                  a.pix_fmt if a.op == 'demodulate' else ingest.picture_format(a.input, a.pix_fmt))
    if header:                                              # a Y4M output's header, written once, before the workers start
        with open(a.output, 'wb') as f:
            f.write(header)
    ranges = [tuple(lo + v for v in frame_range(hi - lo, r, len(a.devices))) for r in range(len(a.devices))]
    if len(a.devices) == 1:
        n = _worker(a, a.devices[0], ranges[0], lo)
    else:
        import multiprocessing as mp
        with mp.get_context('spawn').Pool(len(a.devices)) as pool:
            n = sum(pool.starmap(_worker, [(a, d, r, lo) for d, r in zip(a.devices, ranges)]))
    print('%s: %d frames' % (a.op, n))
    return 0


if __name__ == '__main__':
    sys.exit(main())
