"""Every kernel the dispatcher can pick, held to the float64 oracle (run with -m gpu).

Which kernel serves a call depends on the input type, the line width, the rows of the launch and the tuning knobs of the
environment (csrc/cm_api.cu: cm_create, plan_*_kernel; the launchers in csrc/cm_*.cu):

* u8 input runs the row encoders (k_qam_encode_row2, k_secam_encode_row2, k_niir_encode2, k_proto_encode_row2) and the
  decoders' u8 row staging; float input (test_gpu_parity.py::test_float_planes_against_oracle) runs neither.  The same kernel
  writes the u8 frame and, when asked through ``out_float``, the float planes before the level map / clipping, so the u8
  path is held here to the 1e-4 / 1e-9 bounds of the float path;
* the team geometry of the row kernels changes at fixed line widths, and past the widest one the multi-row kernels serve
  the line: the sweep takes the largest width below each boundary and the boundary itself, and lines up to 3840 samples;
* one row per CTA below 16 x SMs rows per launch, two above (cm_host.h: cm_rows_per_cta), any number through CM_RPC;
* the knobs of cm_create either only reschedule the same arithmetic (byte-identical outputs) or select other kernels
  (same oracle bounds).

A width that no kernel serves must be refused with an error naming the limit; DESIGN.md lists those widths (REFUSED)."""
import functools
import itertools

import numpy as np
import pytest

import conditioning
import oracle
from oracle import frame as oframe
from cases import GOLDEN_CASES, case_id, load_golden
from product import BUILT_KINDS, make_modem
from test_gpu_edges import MAKERS, _lsb
from test_gpu_parity import NIIR_WIDE, _make_or_skip
from color_modem_b200 import comb
from color_modem_b200.color import mac
from color_modem_b200.line import LineConfig, LineStandard as LS
from color_modem_b200.synth import synth_frames_u8

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-4
FP64_TOL = 1e-9

# MAKERS plus the second D2-MAC variant (720-sample composite): oracle kind, preset, line standard, constructor
KINDS = {k: (k,) + v for k, v in MAKERS.items()}
KINDS['mac7'] = ('mac', 'D2MAC_7MHZ', 'GERBER_625', lambda lc: mac.MacModem(lc, mac.MacVariant.D2MAC_7MHZ))


def _is_composed(m):
    """SimpleCombModem / Simple3DCombModem run line by line over their backend (comb.py): u8 frames only on decode."""
    return isinstance(m, comb.SimpleCombModem) and m._impl is None


def _niir_singular(kind, w):
    """NIIR lines sampled much above 13.5 MHz have samples where the hue is decided by float64 rounding (test_gpu_parity.py:
    NIIR_WIDE; DESIGN.md section 6).  From about 1460 samples per line the conditioning probe of the oracle
    (tests/conditioning.py) relaxes more than 0.1 % of the samples (0.10-0.17 % at 1464, 1468, 1924, 1976 and 2164 samples),
    and three noise trials do not find every such sample: the decoded planes are held to quantiles there instead (below)."""
    return kind in ('niir', 'niir_hue') and w >= 1400


def _assert_niir_wide(out_u8, ref_u8, out_f, ref_f, precision, tag):
    """99.9 % of the samples within +-1 LSB and within 1e-4 (fp32) / 1e-8 (fp64) of the oracle; every sample within 3e-2
    (fp32: the hue flips at a singular sample, measured up to 7 LSB at 2560 samples per line) / 1e-6 (fp64)."""
    d = np.abs(out_u8.astype(np.int32) - ref_u8.astype(np.int32))
    assert (d > 1).mean() <= 1e-3, '%s: %.3f %% of the u8 samples off by more than 1 LSB' % (tag, 100 * (d > 1).mean())
    err = np.abs(out_f - ref_f)
    q, top = (FP32_TOL, 3e-2) if precision == 'fp32' else (1e-8, 1e-6)
    assert np.quantile(err, 0.999) <= q and err.max() <= top, '%s: p99.9 %.2e, max %.2e' % (
        tag, np.quantile(err, 0.999), err.max())


def _assert_encode_close(comp, comp_ref, precision, what):
    err = float(np.abs(comp - comp_ref).max())
    assert err <= (FP32_TOL if precision == 'fp32' else FP64_TOL), '%s: composite off by %.2e' % (what, err)


def _assert_decode_close(out, out_ref, precision, singular, bound, what):
    """bound: the fp32 per-sample bound of tests/conditioning.py (a callable, evaluated only for fp32)."""
    err = np.abs(out - out_ref)
    tol = FP32_TOL if precision == 'fp32' else FP64_TOL
    if singular:
        assert np.quantile(err, 0.999) <= tol and err.max() <= (1e-2 if precision == 'fp32' else 1e-6), \
            '%s: p99.9 %.2e, max %.2e' % (what, np.quantile(err, 0.999), err.max())
    elif precision == 'fp32':
        b = bound()
        assert (err <= b).all(), '%s: max excess %.2e at %s' % (what, (err - b).max(),
                                                                 np.unravel_index((err - b).argmax(), err.shape))
    else:
        assert err.max() <= tol, '%s: decoded planes off by %.2e' % (what, err.max())


def _float_dtype(precision):
    import torch
    return torch.float32 if precision == 'fp32' else torch.float64


def _encode(m, rgb, first, precision):
    """u8 frames in, u8 composite and float composite out of the same call."""
    import torch
    x = torch.from_numpy(np.ascontiguousarray(rgb)).cuda()
    n, h = rgb.shape[:2]
    cu = torch.empty((n, h, m.composite_width), dtype=torch.uint8, device='cuda')
    cf = torch.empty((n, h, m.composite_width), dtype=_float_dtype(precision), device='cuda')
    m.encode_frames(x, first, out=cu, out_float=cf)
    return cu.cpu().numpy(), cf.double().cpu().numpy()


def _decode(m, comp_u8, first, precision):
    import torch
    c = torch.from_numpy(np.ascontiguousarray(comp_u8)).cuda()
    n, h = comp_u8.shape[:2]
    ou = torch.empty((n, h, m.output_width, 3), dtype=torch.uint8, device='cuda')
    of = torch.empty((n, h, m.output_width, 3), dtype=_float_dtype(precision), device='cuda')
    m.decode_frames(c, first, out=ou, out_float=of)
    return ou.cpu().numpy(), of.double().cpu().numpy()


# ------------------------------------------------------------------------------------------------------------
# 1. The u8 entry points at float precision, on every golden case
# ------------------------------------------------------------------------------------------------------------
CASES = [c for c in GOLDEN_CASES if c.kind in BUILT_KINDS]


@pytest.mark.parametrize('precision', ['fp32', 'fp64'])
@pytest.mark.parametrize('c', CASES, ids=case_id)
def test_u8_kernels_at_float_precision(c, precision, cuda_required):
    import torch
    g = load_golden(c)
    rgb = synth_frames_u8(1, c.height, c.width, first_frame=c.frame, seed=c.seed, kind=c.content)
    om = oracle.build(oracle.ModemSpec(c.kind, c.variant, c.width, c.height, c.standard, c.chroma_avg, c.notch, c.opt))
    m = make_modem(c, precision)
    comp_u8, comp_f = _make_or_skip(c, precision, lambda: _encode(m, rgb, c.frame, precision))
    # asking for the float planes must not change the path: the u8 frame equals that of a u8-only call
    assert np.array_equal(comp_u8, m.encode_frames(torch.from_numpy(rgb).cuda(), c.frame).cpu().numpy())
    _assert_encode_close(comp_f[0], om.encode(c.frame, rgb[0] / 255.0), precision, 'encode')
    comp_in = oframe.composite_unlevel(g['comp_u8'] / 255.0)
    if _is_composed(m):
        with pytest.raises(NotImplementedError):
            m.decode_frames(torch.from_numpy(g['comp_u8'][None]).cuda(), c.frame,
                            out_float=torch.empty((1, c.height, m.output_width, 3), dtype=_float_dtype(precision),
                                                  device='cuda'))
        return
    out_u8, out_f = _make_or_skip(c, precision, lambda: _decode(m, g['comp_u8'][None], c.frame, precision))
    assert np.array_equal(out_u8, m.decode_frames(torch.from_numpy(g['comp_u8'][None]).cuda(), c.frame).cpu().numpy())
    out_ref = om.decode(c.frame, comp_in)
    _assert_decode_close(out_f[0], out_ref, precision, (c.kind, c.width) in NIIR_WIDE,
                         lambda: conditioning.fp32_bound(lambda x: om.decode(c.frame, x), comp_in, out_ref, FP32_TOL),
                         'decode')


# ------------------------------------------------------------------------------------------------------------
# Oracle reference of a (kind, width, height) batch, built once: the float composite, the oracle's own u8 composite (the
# input of every decode below, so that decode references do not depend on the GPU), the float RGB and the fp32 bound.
# ------------------------------------------------------------------------------------------------------------
class _Ref(object):
    def __init__(self, kind, w, h, first, n, seed):
        okind, variant, std, self.make = KINDS[kind]
        self.kind, self.w, self.h, self.first, self.n = kind, w, h, first, n
        self.lc = LineConfig((w, h), getattr(LS, std))
        self.om = om = oracle.build(oracle.ModemSpec(okind, variant, w, h, std))
        self.rgb = synth_frames_u8(n, h, w, first_frame=first, seed=seed)
        self.comp_f = np.stack([om.encode(first + i, self.rgb[i] / 255.0) for i in range(n)])
        self.comp_u8 = oframe.to_u8(oframe.composite_level(self.comp_f))
        self.comp_in = oframe.composite_unlevel(self.comp_u8 / 255.0)
        self.out_f = np.stack([om.decode(first + i, self.comp_in[i]) for i in range(n)])
        self.out_u8 = oframe.to_u8(self.out_f)
        self._bounds = {}

    def bound(self, i):
        if i not in self._bounds:
            self._bounds[i] = conditioning.fp32_bound(lambda x: self.om.decode(self.first + i, x), self.comp_in[i],
                                                      self.out_f[i], FP32_TOL)
        return self._bounds[i]

    def modem(self, precision='fp32'):
        m = self.make(self.lc)
        return m if precision == 'fp32' else comb._fp64_twin(m)

    def check(self, comp_u8, comp_f, out_u8, out_f, precision='fp32', frames=None, what=''):
        """Outputs of the whole batch (decoded from the oracle's u8 composite): u8 within +-1 LSB of the oracle's frame
        functions, float planes within the 1e-4 / 1e-9 bounds; `frames`: the batch positions to check (default all)."""
        for i in range(self.n) if frames is None else frames:
            tag = '%s %s w=%d h=%d frame %d %s' % (self.kind, precision, self.w, self.h, self.first + i, what)
            assert _lsb(comp_u8[i], self.comp_u8[i]) <= 1, tag + ': u8 composite'
            _assert_encode_close(comp_f[i], self.comp_f[i], precision, tag)
            if _niir_singular(self.kind, self.w):
                _assert_niir_wide(out_u8[i], self.out_u8[i], out_f[i], self.out_f[i], precision, tag)
            else:
                assert _lsb(out_u8[i], self.out_u8[i]) <= 1, tag + ': u8 RGB'
                _assert_decode_close(out_f[i], self.out_f[i], precision, False, lambda: self.bound(i), tag)


@functools.lru_cache(maxsize=None)
def _ref(kind, w, h, first=3, n=2, seed=17):
    try:
        return _Ref(kind, w, h, first, n, seed)
    except ValueError as e:          # a preset whose filter design fails at this sampling rate (scipy), as in test_gpu_widths
        pytest.skip('reference design does not exist at this sampling rate: %s' % e)


def _run(m, ref, precision='fp32'):
    comp_u8, comp_f = _encode(m, ref.rgb, ref.first, precision)
    out_u8, out_f = _decode(m, ref.comp_u8, ref.first, precision)
    return comp_u8, comp_f, out_u8, out_f


# ------------------------------------------------------------------------------------------------------------
# 2. Width sweep
# ------------------------------------------------------------------------------------------------------------
# First width of each team geometry / of the multi-row fallback, from the planners of csrc/cm_api.cu (encoder, decoder)
BOUNDARIES = {
    'ntsc': (736, 1468, 1976, 800, 1596, 2104),            # k_qam_encode_row2 2 / 3 / multi-row; k_qam_bs_row2 2 / 3 / k_qam_bandsplit
    'pal_s': (736, 1468, 1980, 800, 1596, 2104),
    'ntsc_comb': (736, 1468, 1976),                        # encoder and k_qam_rows2 change together
    'ntsc_3d': (736, 1468, 1976),
    'pal_d': (736, 1468, 1980),
    'pal_3d': (736, 1468, 1980),
    'niir': (736, 1468, 1980, 832, 2168),                  # k_niir_encode2 2 / 3 / multi-row; k_niir_decode2 3 / multi-row
    'niir_hue': (736, 1468, 1980, 832, 2168),
    'protosecam': (828, 2052),                             # k_proto_decode2 / encode_row2 geometry 3, multi-row
    'secam': (752, 1924, 2000),                            # k_secam_decode2 geometry 3; row encoder up to 1920; multi-row
}
WIDE = (724, 1924, 2048, 2200, 2560, 3072, 3840)
# MAC: constant-bank taps (960: 3/4, 3/8; 1920), run-time polyphase (720, 1680: 3/7), general resampler (1008: 5/7),
# 2160 (1/3, 1/6) and 3840 (3/16, 3/32, 641 taps); other widths need resamplers the design does not allow
MAC_WIDTHS = (720, 960, 1008, 1680, 1920, 2160, 3840)

# (kind, width) that no kernel serves: refused when the modem is created or on its first call, with the limit named.
# DESIGN.md section 0 ("Limits") lists the same set.
REFUSED = {(k, w): 'line too wide for the NIIR decode kernel' for k in ('niir', 'niir_hue') for w in (3072, 3840)}

SWEEP = sorted({(k, w) for k, bs in BOUNDARIES.items() for b in bs for w in (b - 4, b)} |
               {(k, w) for k in BOUNDARIES for w in WIDE} |
               {(k, w) for k in ('mac', 'mac7') for w in MAC_WIDTHS})


@pytest.mark.parametrize('kind,w', SWEEP, ids=['%s-%d' % kw for kw in SWEEP])
def test_width_sweep(kind, w, cuda_required):
    for h in (7, 12):
        ref = _ref(kind, w, h)
        m = ref.modem('fp32')
        if (kind, w) in REFUSED:
            with pytest.raises(RuntimeError, match=REFUSED[(kind, w)]):
                _run(m, ref)
            return
        ref.check(*_run(m, ref))
        if w <= 2200:
            m64 = ref.modem('fp64')
            try:
                res = _run(m64, ref, 'fp64')
            except RuntimeError as e:
                assert 'too wide' in str(e), e          # the fp64 verification build may not fit shared memory
                continue
            ref.check(*res, precision='fp64')


# ------------------------------------------------------------------------------------------------------------
# 3. Rows per CTA
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('h', [3, 7, 35])
@pytest.mark.parametrize('kind', sorted(MAKERS))
def test_rows_per_cta(kind, h, cuda_required, monkeypatch):
    """1, 2 or 3 rows per CTA (the next row prefetched while one is filtered), where a CTA's last rows are missing: the
    same bytes and floats, within the oracle bounds."""
    ref = _ref(kind, 720, h, first=5, n=3)
    base = None
    for rpc in ('1', '2', '3'):
        monkeypatch.setenv('CM_RPC', rpc)            # read once per handle: a fresh modem per setting
        res = _run(ref.modem(), ref)
        if base is None:
            ref.check(*res, what='CM_RPC=1')
            base = res
        else:
            for a, b in zip(base, res):
                assert np.array_equal(a, b), 'CM_RPC=%s' % rpc


@pytest.mark.parametrize('kind', ['pal_d', 'secam'])
def test_two_rows_per_cta_by_default(kind, cuda_required):
    """A launch of more than 16 x SMs rows takes two rows per CTA without any knob: first, middle and last frame against
    the oracle, every frame byte-equal to the same frame encoded / decoded alone (one row per CTA)."""
    import ctypes as C
    import torch
    from color_modem_b200 import _native as N
    sms = C.c_int(0)
    N.check(N.load().cm_device_info(C.byref(sms), None, None))
    h, w, first = 35, 720, 9
    n = 16 * sms.value // h + 2
    assert n * h > 16 * sms.value
    ref = _ref(kind, w, h, first=first, n=n, seed=29)
    m = ref.modem()
    comp_u8, comp_f, out_u8, out_f = _run(m, ref)
    ref.check(comp_u8, comp_f, out_u8, out_f, frames=(0, n // 2, n - 1), what='of a %d-frame batch' % n)
    for i in range(n):
        one = m.encode_frames(torch.from_numpy(ref.rgb[i:i + 1]).cuda(), first + i).cpu().numpy()
        assert np.array_equal(one[0], comp_u8[i]), ('encode', i)
        one = m.decode_frames(torch.from_numpy(ref.comp_u8[i:i + 1]).cuda(), first + i).cpu().numpy()
        assert np.array_equal(one[0], out_u8[i]), ('decode', i)


# ------------------------------------------------------------------------------------------------------------
# 4. Tuning knobs
# ------------------------------------------------------------------------------------------------------------
def _set(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)


@pytest.mark.parametrize('w', [720, 1920])
@pytest.mark.parametrize('kind', ['ntsc_3d', 'pal_d', 'pal_3d'])
def test_overlapped_passes_are_invisible(kind, w, cuda_required, monkeypatch):
    """CM_OVERLAP runs pass 2 of one chunk on a second stream under pass 1 of the next: the same bytes as one pass pair."""
    import torch
    ref = _ref(kind, w, 12, first=2, n=9)
    c = torch.from_numpy(ref.comp_u8).cuda()
    want = ref.modem().decode_frames(c, 2).cpu().numpy()
    _set(monkeypatch, {'CM_OVERLAP': '1', 'CM_CHUNK': '2'})
    assert np.array_equal(ref.modem().decode_frames(c, 2).cpu().numpy(), want)


HOST_KNOBS = [{'CM_HOST_ROLES': r, 'CM_HOST_CHUNK': c} for r, c in itertools.product(('0', '1'), ('1', '7'))]


@pytest.mark.parametrize('pix_fmt', [None, 'yuv420p'])
@pytest.mark.parametrize('w', [720, 1920])
@pytest.mark.parametrize('kind', ['ntsc_3d', 'pal_d', 'secam'])
def test_host_pipeline_knobs_are_invisible(kind, w, pix_fmt, cuda_required, monkeypatch):
    """Streams per role and frames per host chunk only reschedule copies and kernels: 17 frames (a ragged last chunk)
    through encode_, decode_ and transcode_frames_host give the default's bytes."""
    from color_modem_b200.pixfmt import frame_shape
    ref = _ref(kind, w, 12, first=4, n=2)
    n, h = 17, 12
    rng = np.random.default_rng(5)
    pic = rng.integers(0, 256, (n,) + frame_shape(pix_fmt, w, h), dtype=np.uint8) if pix_fmt else \
        synth_frames_u8(n, h, w, first_frame=4, seed=31)

    def run():
        m = ref.modem()
        comp = m.encode_frames_host(pic, 4, pix_fmt=pix_fmt)
        out = m.decode_frames_host(comp, 4, pix_fmt=pix_fmt)
        tc, to = m.transcode_frames_host(pic, 4, pix_fmt=pix_fmt)
        return comp, out, tc, to

    want = run()
    assert np.array_equal(want[0], want[2]) and np.array_equal(want[1], want[3])
    for env in HOST_KNOBS:
        _set(monkeypatch, env)
        for a, b, what in zip(run(), want, ('encode', 'decode', 'transcode composite', 'transcode picture')):
            assert np.array_equal(a, b), (env, what)


@pytest.mark.parametrize('w', [720, 1920])
@pytest.mark.parametrize('kind', ['mac', 'mac7'])
def test_mac_threads_are_invisible(kind, w, cuda_required, monkeypatch):
    ref = _ref(kind, w, 12)
    want = _run(ref.modem(), ref)
    ref.check(*want)
    for t in ('32', '64', '256'):
        monkeypatch.setenv('CM_MAC_THREADS', t)
        for a, b in zip(_run(ref.modem(), ref), want):
            assert np.array_equal(a, b), t


ORACLE_KNOBS = [('rows_v1', {'CM_ROWS_V1': '1'}), ('min_warps1', {'CM_MIN_WARPS': '1'}),
                ('min_warps4', {'CM_MIN_WARPS': '4'}), ('min_warps8', {'CM_MIN_WARPS': '8'}),
                ('rows_v1_min_warps1', {'CM_ROWS_V1': '1', 'CM_MIN_WARPS': '1'}),
                ('rows_v1_min_warps8', {'CM_ROWS_V1': '1', 'CM_MIN_WARPS': '8'})]


@pytest.mark.parametrize('knob,env', ORACLE_KNOBS, ids=[k[0] for k in ORACLE_KNOBS])
@pytest.mark.parametrize('w', [720, 1920])
@pytest.mark.parametrize('kind', sorted(KINDS))
def test_kernel_selecting_knobs_meet_the_oracle(kind, w, knob, env, cuda_required, monkeypatch):
    """CM_ROWS_V1 (the round-1 multi-row kernels instead of the row kernels) and CM_MIN_WARPS (warps per CTA of the
    multi-row kernels) select other kernels: the same bounds as the default path."""
    ref = _ref(kind, w, 12)
    _set(monkeypatch, env)
    ref.check(*_run(ref.modem(), ref), what=knob)


@pytest.mark.parametrize('w', [960, 1920])
@pytest.mark.parametrize('kind', ['mac', 'mac7'])
def test_mac_shared_memory_taps_meet_the_oracle(kind, w, cuda_required, monkeypatch):
    """CM_MAC_SMEM_TAPS: the resampler taps from the shared-memory table instead of the constant bank."""
    ref = _ref(kind, w, 12)
    monkeypatch.setenv('CM_MAC_SMEM_TAPS', '1')
    ref.check(*_run(ref.modem(), ref), what='CM_MAC_SMEM_TAPS')
