"""The PAL-D decoder's pass 1 as a matrix, from the float64 oracle, and how well the tensor-core kernel can represent it.

For one row, the planes (a', b', LPpre a', LPpre b') of the PAL-D decoder are a linear map of the composite row, with the
carrier at phase 0 for a' and a quarter turn for b' (the row's own phase is a rotation applied afterwards).  This script
pushes the W unit impulses through the oracle (extract -> _am(., 0) / _am(., pi/2) -> pre_lp), reports the band of the
matrix, checks linearity, and evaluates the two-term FP16 split that k_pald_mma (color_modem_b200/csrc/cm_pald_mma.cu)
multiplies with on random u8 rows.  With --library it also compares the library's own matrix (cm_pald_matrix, built on
the host from the handle's filters; needs the built library and a GPU for the handle).

    python tools/pald_matrix.py [--variant PAL] [--standard GERBER_625] [--width 720] [--library]
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle  # noqa: E402

KPRE, KW, TS = 96, 160, 32        # the compiled window of k_pald_mma (cm_host.h: CM_PALD_*)


def oracle_matrix(w, h=576, variant='PAL', standard='GERBER_625'):
    """M[i, 4 x + plane]: plane (a', b', LPpre a', LPpre b') of sample x for a unit impulse at input i."""
    m = oracle.build(oracle.ModemSpec('pal_d', variant, w, h, standard))
    ex = m.qam.extract(np.eye(w))
    a, b = m._am(ex, 0.0), m._am(ex, 0.5 * np.pi)
    planes = np.stack([a, b, m.qam.pre_lp(a), m.qam.pre_lp(b)], axis=-1)    # [i, x, plane]
    return planes.reshape(w, 4 * w), m


def band(M, rel=2.0 ** -26):
    """(lo, hi): output x depends on the inputs [x - lo, x + hi] to `rel` of the largest coefficient of its plane."""
    w = M.shape[0]
    lo = hi = 0
    for p in range(4):
        P = M[:, p::4]
        i, x = np.nonzero(np.abs(P) > rel * np.abs(P).max())
        lo, hi = max(lo, int((x - i).max())), max(hi, int((i - x).max()))
    return lo, hi


def fp16_split_error(M, rows=256, seed=1):
    """Largest difference between the exact planes and those of the kernel's arithmetic (window, column scale, hi + lo)."""
    w = M.shape[0]
    Mu = M * (5.0 / 765.0)
    i = np.arange(w)[:, None]
    x0 = (np.arange(4 * w)[None, :] // 4) // TS * TS
    R = np.where((i >= x0 - KPRE) & (i < x0 - KPRE + KW), Mu, 0.0)
    s = 2.0 ** np.floor(np.log2(1000.0 / np.abs(R).max(axis=0, keepdims=True).clip(1e-300)))
    hi = (R * s).astype(np.float16).astype(np.float64)
    lo = (R * s - hi).astype(np.float16).astype(np.float64)
    X = np.random.default_rng(seed).integers(0, 256, size=(rows, w)).astype(np.float32)
    got = ((X @ hi.astype(np.float32)) + (X @ lo.astype(np.float32))).astype(np.float64) / s
    exact = X.astype(np.float64) @ Mu
    return float(np.abs(got - exact).max()), float(np.abs(exact).max())


def library_matrix(w, h=576, variant='PAL', standard='GERBER_625'):
    import ctypes as C
    from color_modem_b200 import _native as N
    from color_modem_b200.color import pal
    from color_modem_b200.line import LineConfig, LineStandard as LS
    modem = pal.PalDModem(LineConfig((w, h), getattr(LS, standard)), getattr(pal.PalVariant, variant))
    M = np.zeros((w, 4 * w))
    bd = (C.c_int * 2)()
    N.check(N.load().cm_pald_matrix(modem._handle(), M.ctypes.data, bd))
    return M, (bd[0], bd[1])


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--variant', default='PAL', choices=('PAL', 'PAL_M', 'PAL_N'))
    ap.add_argument('--standard', default='GERBER_625', help='line standard (PAL_M: NTSC_525)')
    ap.add_argument('--width', type=int, default=720)
    ap.add_argument('--library', action='store_true', help='compare with the library matrix (needs a GPU)')
    a = ap.parse_args()
    M, m = oracle_matrix(a.width, variant=a.variant, standard=a.standard)
    x = np.random.default_rng(0).uniform(0, 1, a.width)
    lin = np.abs(x @ M[:, 0::4] - m._am(m.qam.extract(x[None]), 0.0)[0]).max()
    lo, hi = band(M)
    err, top = fp16_split_error(M)
    print('%s (%s) width %d: linearity %.1e, band [x - %d, x + %d] at 2^-26 (window [x - %d, x + %d]), fp16 x2 error %.2e '
          '(planes up to %.2f)' % (a.variant, a.standard, a.width, lin, lo, hi, KPRE, KW - KPRE - TS, err, top))
    if a.library:
        L, bd = library_matrix(a.width, variant=a.variant, standard=a.standard)
        print('library: band [x - %d, x + %d], largest difference from the oracle %.2e' % (bd[0], bd[1],
                                                                                          np.abs(L - M).max()))


if __name__ == '__main__':
    main()
