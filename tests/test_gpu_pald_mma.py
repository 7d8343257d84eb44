"""PAL-D decoding on the tensor cores (k_pald_mma, csrc/cm_pald_mma.cu), held to the float64 oracle and to the two-pass
kernels it replaces (run with -m gpu).

The kernel serves float32 handles of PAL-D with u8 composite input and default knobs, where the band of the pass-1 matrix
fits its window (csrc/cm_api.cu: plan_pald_mma).  Each test checks which path ran from the kernel timers: the fused
kernel is timed as CM_K_PALD and leaves CM_K_DECODE_OTHER (pass 2 of the two-pass decoder) empty."""
import ctypes as C
import functools

import numpy as np
import pytest

import conditioning
import oracle
from oracle import frame as oframe
from oracle import modems as omodems, presets
from cases import case_id, load_golden
from product import make_modem
from test_gpu_dispatch import CASES, FP32_TOL, _assert_decode_close, _decode, _ref
from test_gpu_edges import _lsb
from color_modem_b200 import _native as N
from color_modem_b200.color import pal
from color_modem_b200.line import LineConfig, LineStandard as LS

pytestmark = pytest.mark.gpu

KPRE, KW, TS = 96, 160, 32          # csrc/cm_host.h: CM_PALD_*
KOUT = 127                          # output rows of a row tile (cm_pald_mma.cu: kOut)
PALD_CASES = [c for c in CASES if c.kind == 'pal_d']

# Bound of the fused kernel's float planes against the oracle, on the rows it writes (every row with a predecessor in its
# field; the two field tops come from the band-split kernel and keep FP32_TOL).  The composite bytes are exact in FP16,
# B is split into hi + lo and accumulated in FP32; the float32 epilogue (rotation, pairing, re-modulation, colour matrix)
# adds a few ulp of the output.  The largest error over every case of this file, measured on an NVIDIA B200 (1000 W
# power limit), is 1.85e-6 (test_foreign_composite[PAL-720-30-square3], output up to 3.0); FUSED_TOL is 4x that, rounded
# up to a power of two (DESIGN.md section 8).
FUSED_TOL = 2.0 ** -17      # 7.6e-6


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


def _oracle_matrix(w, h, variant='PAL', std='GERBER_625'):
    om = oracle.build(oracle.ModemSpec('pal_d', variant, w, h, std))
    ex = om.qam.extract(np.eye(w))
    a, b = om._am(ex, 0.0), om._am(ex, 0.5 * np.pi)
    return np.stack([a, b, om.qam.pre_lp(a), om.qam.pre_lp(b)], axis=-1).reshape(w, 4 * w)


STANDARD = {'PAL': 'GERBER_625', 'PAL_M': 'NTSC_525', 'PAL_N': 'GERBER_625'}


@pytest.mark.parametrize('variant,w', [('PAL', 720), ('PAL', 736), ('PAL_M', 544), ('PAL_N', 544)],
                         ids=['720', '736', 'PAL_M-544', 'PAL_N-544'])
def test_library_matrix_is_the_oracle_map(variant, w, cuda_required):
    """The matrix the host builds from the handle's filters (cm_pald_matrix) is the oracle's pass-1 map of unit impulses."""
    m = pal.PalDModem(LineConfig((w, 12), getattr(LS, STANDARD[variant])), getattr(pal.PalVariant, variant))
    L = np.zeros((w, 4 * w))
    N.check(N.load().cm_pald_matrix(m._handle(), L.ctypes.data, None))
    M = _oracle_matrix(w, 12, variant, STANDARD[variant])
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
    if fused:
        _assert_fused_close(out_f[0], out_ref, 'decode')
    else:
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
        _assert_fused_close(out_f[i], ref.out_f[i], 'frame %d' % i)


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
        if fused:
            _assert_fused_close(out_f[i], ref.out_f[i], 'w=%d frame %d' % (w, i))
        else:
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


# ------------------------------------------------------------------------------------------------------------
# Shared checks
# ------------------------------------------------------------------------------------------------------------
def _assert_fused_close(out_f, ref_f, what):
    """Float planes of a whole-frame decode served by the fused kernel: FUSED_TOL on the rows it wrote (2 .. H - 1),
    FP32_TOL on the two field tops (the band-split kernel)."""
    err = np.abs(out_f[2:] - ref_f[2:]).max() if out_f.shape[0] > 2 else 0.0
    assert err <= FUSED_TOL, '%s: fused rows off by %.3e' % (what, err)
    top = np.abs(out_f[:2] - ref_f[:2]).max()
    assert top <= FP32_TOL, '%s: field tops off by %.3e' % (what, top)


class _Dec(object):
    """The oracle's decode of a u8 composite batch: float RGB before clipping, u8 RGB, and the per-frame fp32 bound."""
    def __init__(self, om, comp_u8, first):
        self.om, self.comp_u8, self.first, self.n = om, comp_u8, first, comp_u8.shape[0]
        self.comp_in = oframe.composite_unlevel(comp_u8 / 255.0)
        self.out_f = np.stack([om.decode(first + i, self.comp_in[i]) for i in range(self.n)])
        self.out_u8 = oframe.to_u8(self.out_f)
        self._bounds = {}

    def bound(self, i):
        if i not in self._bounds:
            self._bounds[i] = conditioning.fp32_bound(lambda x: self.om.decode(self.first + i, x), self.comp_in[i],
                                                      self.out_f[i], FP32_TOL)
        return self._bounds[i]


def _check_batch(m, ref, monkeypatch, make, fused_expected, what):
    """Decode ref.comp_u8 on `m`: the path the planner promised, +-1 LSB and the float bound against the oracle, and when
    fused, agreement with the two-pass kernels (FP32_TOL, +-1 LSB).  Returns (u8, float) frames."""
    out_u8, out_f, fused = _decode_timed(m, ref.comp_u8, ref.first)
    assert fused == fused_expected, (what, _band(m))
    for i in range(ref.n):
        tag = '%s frame %d' % (what, ref.first + i)
        assert _lsb(out_u8[i], ref.out_u8[i]) <= 1, tag
        if fused:
            _assert_fused_close(out_f[i], ref.out_f[i], tag)
        else:
            _assert_decode_close(out_f[i], ref.out_f[i], 'fp32', False, lambda: ref.bound(i), tag)
    if fused:
        base_u8, base_f, base_fused = _decode_timed(_two_pass(make, monkeypatch), ref.comp_u8, ref.first)
        assert not base_fused
        assert _lsb(out_u8, base_u8) <= 1, what
        assert np.abs(out_f - base_f).max() <= FP32_TOL, what
    return out_u8, out_f


# ------------------------------------------------------------------------------------------------------------
# Every kind of handle the planner serves
# ------------------------------------------------------------------------------------------------------------
# Line widths chosen by rule from the band (lo, hi) of the pass-1 matrix (tools/pald_matrix.py --variant --standard
# --width; the same band as cm_pald_matrix), per variant: the narrowest width whose filter design exists, every width
# whose band sits on the edge of the window (hi == 32 or lo >= 94), the widest served width and the first refused one,
# a refused width inside the served range, and one width with W % 32 == 4 (a last column tile of four samples).
#   PAL (GERBER_625):   452, 456 (60, 33) refused; 460 .. 784 served; hi == 32 at 460 .. 480, 572, 576;
#                       lo >= 94 at 764 .. 784; 788 (97, 29) refused
#   PAL_M (NTSC_525):   384 .. 548 served except 392 (70, 33); hi == 32 at 384, 388, 396 .. 420; lo >= 94 at 536 .. 548;
#                       552 (97, 31) refused
#   PAL_N (GERBER_625): 384 .. 548 served; hi == 32 at 384 .. 420; lo >= 94 at 536 .. 548; 552 (97, 31) refused
EDGE_WIDTHS = {
    'PAL': (452, 456, 460, 464, 468, 472, 476, 480, 572, 576, 612, 764, 768, 772, 776, 780, 784, 788),
    'PAL_M': (384, 388, 392, 396, 400, 404, 408, 412, 416, 420, 452, 536, 540, 544, 548, 552),
    'PAL_N': (384, 388, 392, 396, 400, 404, 408, 412, 416, 420, 452, 536, 540, 544, 548, 552),
}
REFUSED_WIDTHS = {'PAL': (452, 456, 788), 'PAL_M': (392, 552), 'PAL_N': (552,)}
EDGE_CASES = [(v, w) for v, ws in sorted(EDGE_WIDTHS.items()) for w in ws]


def _maker(kind, variant, w, h):
    lc = LineConfig((w, h), getattr(LS, STANDARD[variant]))
    pv = getattr(pal.PalVariant, variant)
    if kind == 'pal_d':
        return lambda: pal.PalDModem(lc, pv)
    return lambda: pal.Pal3DModem(lc, pv, use_sin=False, use_cos=False)


@functools.lru_cache(maxsize=None)
def _variant_ref(variant, w, h, first=3, n=2, seed=17):
    """Oracle reference of a PAL-D batch of `variant` (encoded by the oracle from synthetic pictures)."""
    from color_modem_b200.synth import synth_frames_u8
    try:
        om = oracle.build(oracle.ModemSpec('pal_d', variant, w, h, STANDARD[variant]))
    except ValueError as e:          # a preset whose filter design fails at this sampling rate (scipy)
        pytest.skip('reference design does not exist at this sampling rate: %s' % e)
    rgb = synth_frames_u8(n, h, w, first_frame=first, seed=seed)
    comp = np.stack([om.encode(first + i, rgb[i] / 255.0) for i in range(n)])
    return _Dec(om, oframe.to_u8(oframe.composite_level(comp)), first)


@pytest.mark.parametrize('kind', ['pal_d', 'pal_3d_plain'])
@pytest.mark.parametrize('variant,w', EDGE_CASES, ids=['%s-%d' % c for c in EDGE_CASES])
def test_every_served_handle(variant, w, kind, cuda_required, monkeypatch):
    """PalDModem and Pal3DModem(use_sin=False, use_cos=False) (plain PAL-D, pal.py:181-182) of PAL, PAL-M and PAL-N at
    the widths above: the fused kernel exactly where the band fits the window, held to the oracle and to the two-pass
    kernels; the two-pass kernels elsewhere."""
    ref = _variant_ref(variant, w, 12)
    if kind == 'pal_3d_plain':       # the oracle of the plain PAL-3D handle is PAL-D's
        o3 = omodems.Pal3D(oracle.ModemSpec('pal_3d', variant, w, 12, STANDARD[variant]), presets.PAL[variant],
                           use_sin=False, use_cos=False)
        assert np.array_equal(np.stack([o3.decode(ref.first + i, ref.comp_in[i]) for i in range(ref.n)]), ref.out_f)
    make = _maker(kind, variant, w, 12)
    m = make()
    assert _fits(m) == (w not in REFUSED_WIDTHS[variant]), (w, _band(m))
    _check_batch(m, ref, monkeypatch, make, _fits(m), '%s %s w=%d' % (kind, variant, w))


# ------------------------------------------------------------------------------------------------------------
# Long row-tile walks, and tile boundaries on frame boundaries
# ------------------------------------------------------------------------------------------------------------
def _sm_count():
    sms = C.c_int(0)
    N.check(N.load().cm_device_info(C.byref(sms), None, None))
    return sms.value


def _walk(n, h, w):
    """(row tiles, row tiles per CTA) of k_pald_mma for n whole frames of h rows (cm_pald_mma.cu: launch_pald_mma): the
    rows 2 .. h - 1 of each frame and the predecessor that opens each field, 127 list rows per tile."""
    out = h - 2
    per_frame = ((out + 1) >> 1) + 1 + ((out >> 1) + 1 if out >> 1 else 0)
    tiles = -(-n * per_frame // KOUT)
    gx = max(1, min(tiles, _sm_count() // -(-w // TS)))
    return tiles, -(-tiles // gx)


def _encoded(n, h, w, first, seed):
    """A composite batch from the library's own encoder (the decode input only needs to be composite)."""
    import torch
    from color_modem_b200.synth import synth_frames_u8
    m = pal.PalDModem(LineConfig((w, h), LS.GERBER_625))
    rgb = synth_frames_u8(n, h, w, first_frame=first, seed=seed)
    return m.encode_frames(torch.from_numpy(rgb).cuda(), first).cpu().numpy()


def _check_walk(n, h, first, monkeypatch, w=720):
    import torch
    comp = _encoded(n, h, w, first, seed=41)
    make = _maker('pal_d', 'PAL', w, h)
    m = make()
    out_u8, out_f, fused = _decode_timed(m, comp, first)
    assert fused
    base_u8, base_f, base_fused = _decode_timed(_two_pass(make, monkeypatch), comp, first)
    assert not base_fused
    assert _lsb(out_u8, base_u8) <= 1
    assert np.abs(out_f - base_f).max() <= FP32_TOL
    om = oracle.build(oracle.ModemSpec('pal_d', 'PAL', w, h, 'GERBER_625'))
    for i in sorted({0, n // 2, n - 1}):
        ref = _Dec(om, comp[i:i + 1], first + i)
        assert _lsb(out_u8[i], ref.out_u8[0]) <= 1, ('frame', i)
        _assert_fused_close(out_f[i], ref.out_f[0], 'frame %d of %d' % (i, n))
    # batch-position invariance: a row is computed from the same bytes with the same B whatever lane, tile or CTA it
    # lands on, so every frame is bit for bit the frame decoded alone at the same absolute frame number
    for i in range(n):
        one_u8 = torch.empty((1, h, w, 3), dtype=torch.uint8, device='cuda')
        one_f = torch.empty((1, h, w, 3), dtype=torch.float32, device='cuda')
        m.decode_frames(torch.from_numpy(comp[i:i + 1]).cuda(), first + i, out=one_u8, out_float=one_f)
        assert np.array_equal(one_u8.cpu().numpy()[0], out_u8[i]), ('u8', i)
        assert np.array_equal(one_f.double().cpu().numpy()[0], out_f[i]), ('float', i)


def test_long_row_tile_walk(cuda_required, monkeypatch):
    """64 frames of 720x576: each CTA walks dozens of row tiles, its two A buffers and accumulators alternating."""
    tiles, per_cta = _walk(64, 576, 720)
    assert per_cta >= 16, (tiles, per_cta)
    _check_walk(64, 576, 11, monkeypatch)


# frames x list rows a multiple of the 127 rows of a tile (h = 127: every tile is one frame, its halo lane the last row
# of the previous frame), one row more or fewer; h = 3 (a predecessor and one output row per frame) and h = 4
@pytest.mark.parametrize('n,h', [(8, 127), (8, 126), (8, 128), (127, 128), (127, 126), (400, 3), (200, 4)])
def test_tile_boundaries_on_frame_boundaries(n, h, cuda_required, monkeypatch):
    tiles, per_cta = _walk(n, h, 720)
    assert tiles >= 6, tiles
    _check_walk(n, h, 2, monkeypatch)


# ------------------------------------------------------------------------------------------------------------
# Composite no encoder produces
# ------------------------------------------------------------------------------------------------------------
IMPULSE_OFFSETS = (0, 1, 7, 8, 95, 96, 127, 128, 159)      # from x0 - KPRE: the K window of a column tile


def _pattern(name, h, w, step):
    """u8 composite [h, w]; step: subcarrier phase per sample (radians)."""
    x = np.arange(w)
    if name == 'random':
        return np.random.default_rng(h * w).integers(0, 256, (h, w), dtype=np.uint8)
    if name in ('flat0', 'flat255'):
        return np.full((h, w), 0 if name == 'flat0' else 255, np.uint8)
    if name.startswith('square'):
        p = int(name[6:])
        return np.tile(np.where(x % p < p // 2, 0, 255).astype(np.uint8), (h, 1))
    if name == 'sine':
        ph = step * x[None, :] + 0.7 * np.arange(h)[:, None]
        return np.rint(127.5 + 127.5 * np.sin(ph)).astype(np.uint8)
    assert name in ('impulse255', 'impulse0')
    # row r carries position (r // 2) % 14 (both fields): one of the K-window offsets in every column tile, or one of
    # the columns 0, W - 4 .. W - 1
    comp = np.full((h, w), 128, np.uint8)
    tiles = np.arange(-(-w // TS)) * TS
    for r in range(h):
        k = (r // 2) % (len(IMPULSE_OFFSETS) + 5)
        xs = tiles - KPRE + IMPULSE_OFFSETS[k] if k < len(IMPULSE_OFFSETS) else \
            np.array([(0, w - 4, w - 3, w - 2, w - 1)[k - len(IMPULSE_OFFSETS)]])
        comp[r, xs[(xs >= 0) & (xs < w)]] = 255 if name == 'impulse255' else 0
    return comp


FOREIGN = [('PAL', 720, h, p) for p, h in (('random', 48), ('flat0', 24), ('flat255', 26), ('square2', 28),
                                            ('square3', 30), ('square4', 34), ('square6', 38), ('sine', 40),
                                            ('impulse255', 32), ('impulse0', 32), ('random', 576))] + \
          [('PAL_M', 544, h, p) for p, h in (('random', 24), ('square2', 24), ('sine', 30), ('impulse255', 32),
                                             ('impulse0', 32))]


@pytest.mark.parametrize('variant,w,h,pattern', FOREIGN, ids=['%s-%d-%d-%s' % c for c in FOREIGN])
def test_foreign_composite(variant, w, h, pattern, cuda_required, monkeypatch):
    """Saturated, noisy, Nyquist-rate and impulse composite: PAL-D decoding is affine in the composite before clipping,
    so the oracle comparison is well conditioned for any bytes (the conditioning probe relaxes no sample, which is what
    makes FUSED_TOL a fair bound).  Both paths against the oracle."""
    om = oracle.build(oracle.ModemSpec('pal_d', variant, w, h, STANDARD[variant]))
    first = 6
    comp = _pattern(pattern, h, w, 2.0 * om.qam.step)[None]
    ref = _Dec(om, comp, first)
    assert (ref.bound(0) == FP32_TOL).all()
    make = _maker('pal_d', variant, w, h)
    _check_batch(make(), ref, monkeypatch, make, True, '%s %d %s' % (variant, w, pattern))
    out_u8, out_f, fused = _decode_timed(_two_pass(make, monkeypatch), comp, first)
    assert not fused
    assert _lsb(out_u8[0], ref.out_u8[0]) <= 1
    _assert_decode_close(out_f[0], ref.out_f[0], 'fp32', False, lambda: ref.bound(0), 'two-pass %s' % pattern)


# ------------------------------------------------------------------------------------------------------------
# u8 row windows through cm_decode_ex
# ------------------------------------------------------------------------------------------------------------
WIN_H = 320
SENT_U8, SENT_F = 0x5a, -7.25


@functools.lru_cache(maxsize=None)
def _whole(first):
    """Three whole 720x320 frames from `first` and their decode on the fused kernel (u8, float)."""
    comp = _encoded(3, WIN_H, 720, first, seed=43)
    m = _maker('pal_d', 'PAL', 720, WIN_H)()
    out_u8, out_f, fused = _decode_timed(m, comp, first)
    assert fused
    return comp, out_u8, out_f.astype(np.float32)


def _decode_window(m, comp, win, first, float_in=False):
    """cm_decode_ex over a row window, outputs pre-filled with a sentinel: (u8, float32, fused)."""
    import torch
    n, nrows, w = comp.shape
    tin = torch.from_numpy(oframe.composite_unlevel(comp / 255.0).astype(np.float32) if float_in else comp).cuda()
    ou = torch.full((n, nrows, w, 3), SENT_U8, dtype=torch.uint8, device='cuda')
    of = torch.full((n, nrows, w, 3), SENT_F, dtype=torch.float32, device='cuda')
    m.timing(True)
    N.check(N.load().cm_decode_ex(m._handle(), C.byref(win), None if float_in else tin.data_ptr(),
                                  tin.data_ptr() if float_in else None, ou.data_ptr(), of.data_ptr(), int(first), n,
                                  torch.cuda.current_stream().cuda_stream))
    fused = m.timing_read(N.K_PALD)[1] > 0 and m.timing_read(N.K_DECODE_OTHER)[1] == 0
    m.timing(False)
    return ou.cpu().numpy(), of.cpu().numpy(), fused


def _outside(out, ob, oc):
    return np.concatenate([out[:, :ob], out[:, ob + oc:]], axis=1)


FIRSTS = (0, 5, 2 ** 31 + 7)


@pytest.mark.parametrize('y0', [0, 1, 37, 300])
@pytest.mark.parametrize('nrows', [3, 5, 12])
def test_u8_row_windows(nrows, y0, cuda_required):
    """Windows cut from whole frames: every output row bit for bit the same line of the whole-frame decode, every other
    row left as it was, u8 and float; the fused kernel serves each call."""
    m = _maker('pal_d', 'PAL', 720, WIN_H)()
    k = 0
    for ob in (2, 3, 5):
        for oc in range(1, nrows - ob + 1):
            for n in (1, 3):
                first = FIRSTS[k % len(FIRSTS)]
                k += 1
                comp, want_u8, want_f = _whole(first)
                win = N.Window(nrows, y0, ob, oc, N.MODE_DEFAULT, 0, 0)
                out_u8, out_f, fused = _decode_window(m, np.ascontiguousarray(comp[:n, y0:y0 + nrows]), win, first)
                tag = (nrows, y0, ob, oc, n, first)
                assert fused, tag
                lines = slice(y0 + ob, y0 + ob + oc)
                assert np.array_equal(out_u8[:, ob:ob + oc], want_u8[:n, lines]), tag
                assert np.array_equal(out_f[:, ob:ob + oc], want_f[:n, lines]), tag
                assert (_outside(out_u8, ob, oc) == SENT_U8).all(), tag
                assert (_outside(out_f, ob, oc) == np.float32(SENT_F)).all(), tag


@pytest.mark.parametrize('nrows,y0,ob,oc', [(3, 0, 2, 1), (5, 1, 3, 2), (12, 37, 2, 10), (12, 300, 5, 4)])
def test_u8_row_windows_with_phase_offset(nrows, y0, ob, oc, cuda_required, monkeypatch):
    """An explicit start phase has no whole-frame equivalent: the fused window agrees with the same window on the
    two-pass kernels and with the float-input window (which never takes the fused path)."""
    make = _maker('pal_d', 'PAL', 720, WIN_H)
    comp = np.ascontiguousarray(_whole(5)[0][:, y0:y0 + nrows])
    win = N.Window(nrows, y0, ob, oc, N.MODE_DEFAULT, 0, 0x3C6EF372FE94F82B)
    out_u8, out_f, fused = _decode_window(make(), comp, win, 5)
    assert fused
    assert (_outside(out_u8, ob, oc) == SENT_U8).all() and (_outside(out_f, ob, oc) == np.float32(SENT_F)).all()
    for name, (b_u8, b_f, b_fused) in (('two-pass', _decode_window(_two_pass(make, monkeypatch), comp, win, 5)),
                                       ('float input', _decode_window(make(), comp, win, 5, float_in=True))):
        assert not b_fused, name
        assert _lsb(out_u8, b_u8) <= 1, name
        assert np.abs(out_f[:, ob:ob + oc] - b_f[:, ob:ob + oc]).max() <= FP32_TOL, name


# ------------------------------------------------------------------------------------------------------------
# Misaligned frames are refused before any launch
# ------------------------------------------------------------------------------------------------------------
def test_misaligned_frames_are_refused(cuda_required):
    """Contiguous views at storage offsets the kernels cannot load from (u8: 32-bit words; float32: 128-bit vectors):
    ValueError in Python, CM_ERR_INVALID from the C ABI, and no kernel launched."""
    import torch
    n, h, w = 2, 12, 720
    m = _maker('pal_d', 'PAL', w, h)()
    m._handle()
    cnt = N.launch_count()

    def view(dtype, shape, offset):
        size = int(np.prod(shape))
        t = torch.zeros(size + 16, dtype=dtype, device='cuda')[offset:offset + size].view(*shape)
        assert t.is_contiguous()
        return t

    comp, rgb = (n, h, w), (n, h, w, 3)
    with pytest.raises(ValueError, match='aligned'):
        m.decode_frames(view(torch.uint8, comp, 1))
    for off in (1, 2, 3):
        with pytest.raises(ValueError, match='aligned'):
            m.decode_frames(view(torch.uint8, comp, 0), out=view(torch.uint8, rgb, off))
        with pytest.raises(ValueError, match='aligned'):
            m.decode_frames(view(torch.uint8, comp, 0), out_float=view(torch.float32, rgb, off))
        with pytest.raises(ValueError, match='aligned'):
            m.encode_frames(view(torch.uint8, rgb, off))
        with pytest.raises(ValueError, match='aligned'):
            m.encode_frames(view(torch.uint8, rgb, 0), out=view(torch.uint8, comp, off))
    lib, st = N.load(), torch.cuda.current_stream().cuda_stream
    good_in, good_out = view(torch.uint8, comp, 0), view(torch.uint8, rgb, 0)
    calls = [(view(torch.uint8, comp, 1).data_ptr(), None, good_out.data_ptr(), None),
             (good_in.data_ptr(), None, view(torch.uint8, rgb, 2).data_ptr(), None),
             (good_in.data_ptr(), None, None, view(torch.float32, rgb, 2).data_ptr()),
             (None, view(torch.float32, comp, 1).data_ptr(), good_out.data_ptr(), None)]
    for args in calls:
        assert lib.cm_decode_ex(m._handle(), None, *args, 0, n, st) == -1, args      # CM_ERR_INVALID
        assert b'aligned' in lib.cm_last_error()
    assert N.launch_count() == cnt
