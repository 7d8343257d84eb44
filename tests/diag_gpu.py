"""Diagnostic (not a test): print CUDA-vs-oracle errors for every built golden case.  Run on the GPU box:
    python tests/diag_gpu.py [kind-substring]"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import oracle                                              # noqa: E402
from oracle import frame as oframe                         # noqa: E402
from cases import GOLDEN_CASES, case_id, load_golden       # noqa: E402
from product import BUILT_KINDS, make_modem                # noqa: E402
from color_modem_b200.synth import synth_frames_u8         # noqa: E402

import torch                                               # noqa: E402

sel = sys.argv[1] if len(sys.argv) > 1 else ''
for c in GOLDEN_CASES:
    if c.kind not in BUILT_KINDS or sel not in case_id(c):
        continue
    g = load_golden(c)
    rgb = synth_frames_u8(1, c.height, c.width, first_frame=c.frame, seed=c.seed, kind=c.content)[0]
    om = oracle.build(oracle.ModemSpec(c.kind, c.variant, c.width, c.height, c.standard, c.chroma_avg, c.notch, c.opt))
    rgb01 = rgb / 255.0
    comp_ref = om.encode(c.frame, rgb01)
    comp_in = oframe.composite_unlevel(g['comp_u8'] / 255.0)
    out_ref = om.decode(c.frame, comp_in)
    line = case_id(c) + ':'
    for prec in ('fp32', 'fp64'):
        try:
            m = make_modem(c, prec)
            ce = np.abs(m.encode_frame_float(rgb01, c.frame) - comp_ref)
            de = np.abs(m.decode_frame_float(comp_in, c.frame) - out_ref)
            line += '  %s enc %.2e dec %.2e (p99.9 %.2e, rows>tol %s)' % (
                prec, ce.max(), de.max(), np.quantile(de, 0.999),
                sorted(set(np.nonzero(de > (1e-4 if prec == 'fp32' else 1e-9))[0]))[:6])
        except Exception as e:                              # noqa: BLE001
            line += '  %s ERROR %s' % (prec, e)
    m = make_modem(c)
    cu = m.encode_frames(torch.from_numpy(rgb[None]).cuda(), first_frame=c.frame)[0].cpu().numpy()
    du = m.decode_frames(torch.from_numpy(g['comp_u8'][None]).cuda(), first_frame=c.frame)[0].cpu().numpy()
    line += '  u8 enc %d dec %d LSB' % (np.abs(cu.astype(int) - g['comp_u8']).max(), np.abs(du.astype(int) - g['rgb_u8']).max())
    print(line, flush=True)
