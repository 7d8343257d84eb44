"""PAL-D decoding on the tensor cores (k_pald_mma, csrc/cm_pald_mma.cu), held to the float64 oracle and to the two-pass
kernels it replaces (run with -m gpu).

The kernel serves float32 handles of PAL-D with u8 composite input and default knobs, where the band of the pass-1 matrix
fits its window (csrc/cm_api.cu: plan_pald_mma).  Each test checks which path ran from the kernel timers: the fused
kernel is timed as CM_K_PALD and leaves CM_K_DECODE_OTHER (pass 2 of the two-pass decoder) empty."""
import ctypes as C

import numpy as np
import pytest

import conditioning
import oracle
from oracle import frame as oframe
from cases import case_id, load_golden
from product import make_modem
from test_gpu_dispatch import CASES, FP32_TOL, _assert_decode_close, _decode, _ref
from test_gpu_edges import _lsb
from color_modem_b200 import _native as N

pytestmark = pytest.mark.gpu

KPRE, KW, TS = 96, 160, 32          # csrc/cm_host.h: CM_PALD_*
PALD_CASES = [c for c in CASES if c.kind == 'pal_d']


def _band(m):
    bd = (C.c_int * 2)()
    N.check(N.load().cm_pald_matrix(m._handle(), None, bd))
    return bd[0], bd[1]


def _fits(m):
    lo, hi = _band(m)
    return lo <= KPRE and hi <= KW - KPRE - TS


def _decode_timed(m, comp_u8, first):
    """(u8 frames, float frames, True when the fused kernel served the call)"""
    m.timing(True)
    out_u8, out_f = _decode(m, comp_u8, first, 'fp32')
    fused = m.timing_read(N.K_PALD)[1] > 0 and m.timing_read(N.K_DECODE_OTHER)[1] == 0
    m.timing(False)
    return out_u8, out_f, fused


def _two_pass(make, monkeypatch):
    monkeypatch.setenv('CM_PALD_MMA', '0')          # read once per handle, when the handle is created
    m = make()
    m._handle()
    monkeypatch.delenv('CM_PALD_MMA')
    return m


def _oracle_matrix(w, h):
    om = oracle.build(oracle.ModemSpec('pal_d', 'PAL', w, h, 'GERBER_625'))
    ex = om.qam.extract(np.eye(w))
    a, b = om._am(ex, 0.0), om._am(ex, 0.5 * np.pi)
    return np.stack([a, b, om.qam.pre_lp(a), om.qam.pre_lp(b)], axis=-1).reshape(w, 4 * w)


@pytest.mark.parametrize('w', [720, 736])
def test_library_matrix_is_the_oracle_map(w, cuda_required):
    """The matrix the host builds from the handle's filters (cm_pald_matrix) is the oracle's pass-1 map of unit impulses."""
    from color_modem_b200.color import pal
    from color_modem_b200.line import LineConfig, LineStandard as LS
    m = pal.PalDModem(LineConfig((w, 12), LS.GERBER_625))
    L = np.zeros((w, 4 * w))
    N.check(N.load().cm_pald_matrix(m._handle(), L.ctypes.data, None))
    M = _oracle_matrix(w, 12)
    assert np.abs(L - M).max() <= 1e-9 * np.abs(M).max()
    lo, hi = _band(m)
    assert 0 < lo <= 120 and 0 < hi <= 40, (lo, hi)


@pytest.mark.parametrize('c', PALD_CASES, ids=case_id)
def test_golden_cases_against_oracle(c, cuda_required):
    """Every PAL-D golden case through out_float: within the fp32 bound of the oracle and +-1 LSB, the u8 frame the same
    as that of a u8-only call."""
    import torch
    g = load_golden(c)
    m = make_modem(c, 'fp32')
    out_u8, out_f, fused = _decode_timed(m, g['comp_u8'][None], c.frame)
    assert fused == (_fits(m) and not c.notch), (c, _band(m))
    assert np.array_equal(out_u8, m.decode_frames(torch.from_numpy(g['comp_u8'][None]).cuda(), c.frame).cpu().numpy())
    om = oracle.build(oracle.ModemSpec(c.kind, c.variant, c.width, c.height, c.standard, c.chroma_avg, c.notch, c.opt))
    comp_in = oframe.composite_unlevel(g['comp_u8'] / 255.0)
    out_ref = om.decode(c.frame, comp_in)
    assert _lsb(out_u8[0], oframe.to_u8(out_ref)) <= 1
    _assert_decode_close(out_f[0], out_ref, 'fp32', False,
                         lambda: conditioning.fp32_bound(lambda x: om.decode(c.frame, x), comp_in, out_ref, FP32_TOL),
                         'decode')


@pytest.mark.parametrize('n,h,first', [(1, 576, 0), (2, 576, 7), (3, 35, 1), (37, 35, 12), (37, 7, 3)])
def test_tiles_across_fields_and_frames(n, h, first, cuda_required, monkeypatch):
    """Row tiles of 127 output rows run across field and frame boundaries: the fused kernel against the two-pass kernels
    on the whole batch (1e-4, +-1 LSB), and against the oracle on its first, middle and last frame."""
    ref = _ref('pal_d', 720, h, first=first, n=n, seed=31)
    out_u8, out_f, fused = _decode_timed(ref.modem(), ref.comp_u8, first)
    assert fused
    base_u8, base_f, base_fused = _decode_timed(_two_pass(ref.modem, monkeypatch), ref.comp_u8, first)
    assert not base_fused
    assert _lsb(out_u8, base_u8) <= 1
    assert np.abs(out_f - base_f).max() <= FP32_TOL
    for i in sorted({0, n // 2, n - 1}):
        assert _lsb(out_u8[i], ref.out_u8[i]) <= 1, ('frame', i)
        _assert_decode_close(out_f[i], ref.out_f[i], 'fp32', False, lambda: ref.bound(i), 'frame %d' % i)


# widths that are not multiples of the 32-sample column tile, and the k_qam_rows2 planner boundary of PAL-D (736) with
# the width below it; wider lines have a band beyond the window and keep the two-pass kernels
@pytest.mark.parametrize('w', [644, 676, 700, 708, 716, 724, 732, 736, 764, 800, 1464, 1468])
def test_widths(w, cuda_required, monkeypatch):
    ref = _ref('pal_d', w, 12, first=3, n=2)
    m = ref.modem()
    out_u8, out_f, fused = _decode_timed(m, ref.comp_u8, ref.first)
    assert fused == _fits(m), (w, _band(m))
    for i in range(ref.n):
        assert _lsb(out_u8[i], ref.out_u8[i]) <= 1
        _assert_decode_close(out_f[i], ref.out_f[i], 'fp32', False, lambda: ref.bound(i), 'w=%d frame %d' % (w, i))
    if fused:
        base_u8, base_f, _ = _decode_timed(_two_pass(ref.modem, monkeypatch), ref.comp_u8, ref.first)
        assert _lsb(out_u8, base_u8) <= 1
        assert np.abs(out_f - base_f).max() <= FP32_TOL


def test_fp64_build_keeps_two_pass_kernels(cuda_required):
    import torch
    ref = _ref('pal_d', 720, 35, first=5, n=3)
    m64 = ref.modem('fp64')
    m64.timing(True)
    m64.decode_frames(torch.from_numpy(ref.comp_u8).cuda(), ref.first)
    assert m64.timing_read(N.K_DECODE_OTHER)[1] > 0
    m64.timing(False)
