"""Small encode->decode of every modem family at 720 and 1920 samples per line, for compute-sanitizer:

    compute-sanitizer --tool memcheck  python tools/sanitize.py
    compute-sanitizer --tool racecheck python tools/sanitize.py
    compute-sanitizer --tool memcheck  python tools/sanitize.py --widths 724,1468,1924,2104,2168,3840 [name]

(few rows, two frames: the kernels' shared-memory choreography is the same at any height).  --widths takes other line
widths, e.g. the geometry boundaries and wide lines of tests/test_gpu_dispatch.py; a family that has no design at a width
(MAC resamplers) or refuses it (too wide for its kernels) is reported and skipped."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch                                                            # noqa: E402
from color_modem_b200.line import LineConfig, LineStandard as LS        # noqa: E402
from color_modem_b200.color import ntsc, pal, secam, niir, protosecam, mac   # noqa: E402
from color_modem_b200 import comb                                        # noqa: E402
from color_modem_b200.synth import synth_frames_u8                       # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument('only', nargs='?', default='', help='run the cases whose name contains this')
ap.add_argument('--widths', default='720,1920', help='comma-separated line widths (default 720,1920)')
args = ap.parse_args()
only = args.only
for w in [int(x) for x in args.widths.split(',')]:
    h = 12
    cases = [('ntsc', lambda: ntsc.NtscModem(LineConfig((w, h), LS.NTSC_525))),
             ('ntsc3d', lambda: comb.Simple3DCombModem(ntsc.NtscCombModem(LineConfig((w, h), LS.NTSC_525)))),
             ('pald', lambda: pal.PalDModem(LineConfig((w, h), LS.GERBER_625))),
             ('pal3d', lambda: pal.Pal3DModem(LineConfig((w, h), LS.GERBER_625))),
             ('secam', lambda: comb.ColorAveragingModem(secam.SecamModem(LineConfig((w, h), LS.GERBER_625), secam.SecamVariant.SECAM_III))),
             ('niir', lambda: niir.HueCorrectingNiirModem(LineConfig((w, h), LS.GERBER_625))),
             ('proto', lambda: comb.ColorAveragingModem(protosecam.ProtoSecamModem(LineConfig((w, h), LS.FRENCH_819)))),
             ('mac7', lambda: mac.MacModem(LineConfig((w, h), LS.GERBER_625), mac.MacVariant.D2MAC_7MHZ)),
             ('mac12', lambda: comb.ColorAveragingModem(mac.MacModem(LineConfig((w, h), LS.GERBER_625))))]
    for name, make in cases:
        if only and only not in name:
            continue
        try:
            m = make()
            rgb = torch.from_numpy(synth_frames_u8(2, h, w, seed=3)).cuda()
            comp = m.encode_frames(rgb, first_frame=5)
            out = m.decode_frames(comp, first_frame=5)
        except (ValueError, RuntimeError) as e:
            print('%s %d: skipped: %s' % (name, w, e), flush=True)
            continue
        torch.cuda.synchronize()
        print('%s %d: ok, checksum %d' % (name, w, int(out.sum().item())), flush=True)
