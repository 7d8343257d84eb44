"""ctypes binding of libcolormodem_b200.so (include/color_modem_b200.h).

There is deliberately no fallback: if the CUDA library is missing or cannot be loaded, importing the modem
classes still works (so filter design can be unit-tested on a CPU box) but creating a handle or running any
modem raises NativeUnavailable.
"""
import ctypes as C
import os

ABI_VERSION = 3
MAX_SECTIONS, MAX_FILTERS, MAX_SCALARS, MAX_RESAMPLERS, MAX_TAPS = 6, 10, 48, 6, 1024

KIND_QAM_BANDSPLIT, KIND_NTSC_COMB, KIND_NTSC_3D, KIND_PAL_D, KIND_PAL_3D = 1, 2, 3, 4, 5
KIND_SECAM, KIND_NIIR, KIND_PROTOSECAM, KIND_MAC = 6, 7, 8, 9

FLAG_PAL_VSWITCH, FLAG_CHROMA_AVG, FLAG_HUE_CORRECT, FLAG_NTSC_NO_COMB = 1, 2, 4, 8
FLAG_PAL3D_SIN, FLAG_PAL3D_COS, FLAG_SECAM_BELL, FLAG_SECAM_LF, FLAG_PROTO_LUMA, FLAG_NOTCH, FLAG_MINAVG = 16, 32, 64, 128, 256, 512, 1024

FP32, FP64 = 0, 1

LIB_NAME = 'libcolormodem_b200.so'
# CM_B200_LIB: tuning aid, load an alternative build of the same library (tools/variants.sh)
LIB_PATH = os.environ.get('CM_B200_LIB') or os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)


class NativeUnavailable(RuntimeError):
    pass


class Filter(C.Structure):
    _fields_ = [('nsec', C.c_int32), ('shift', C.c_int32), ('n', C.c_int32), ('rate', C.c_int32),
                ('sos', (C.c_double * 5) * MAX_SECTIONS)]


class Resampler(C.Structure):
    _fields_ = [('up', C.c_int32), ('down', C.c_int32), ('half', C.c_int32), ('ntaps', C.c_int32),
                ('taps', C.c_double * MAX_TAPS)]


class Desc(C.Structure):
    _fields_ = [('abi_version', C.c_int32), ('kind', C.c_int32), ('flags', C.c_int32),
                ('width', C.c_int32), ('height', C.c_int32), ('comp_width', C.c_int32), ('out_width', C.c_int32),
                ('digital_shift', C.c_int32), ('odd_first', C.c_int32), ('even_first', C.c_int32),
                ('ref_line', C.c_int32), ('frame_cycle', C.c_int32),
                ('frame_shift_turns', C.c_uint64), ('line_shift_turns', C.c_uint64),
                ('phases', C.c_uint64 * 16),
                ('scalars', C.c_double * MAX_SCALARS),
                ('enc_matrix', C.c_double * 9), ('dec_matrix', C.c_double * 9),
                ('nfilters', C.c_int32), ('filters', Filter * MAX_FILTERS),
                ('nresamplers', C.c_int32), ('resamplers', Resampler * MAX_RESAMPLERS)]


class Window(C.Structure):
    _fields_ = [('nrows', C.c_int32), ('y0', C.c_int32), ('out_begin', C.c_int32), ('out_count', C.c_int32),
                ('mode', C.c_int32), ('reserved', C.c_int32), ('phase_offset', C.c_uint64)]


MODE_DEFAULT, MODE_BANDSPLIT_NOSTRIP, MODE_EXTRACT_CHROMA = 0, 1, 2


class PixFmt(C.Structure):
    _fields_ = [('format', C.c_int32), ('matrix', C.c_int32), ('range', C.c_int32), ('reserved', C.c_int32)]


PIX_RGB24, PIX_YUV420P = 0, 1
YUV_BT601, YUV_BT709 = 0, 1
YUV_LIMITED, YUV_FULL = 0, 1


EXPORTS = ['cm_abi_version', 'cm_sizeof_desc', 'cm_last_error', 'cm_device_info', 'cm_create', 'cm_destroy', 'cm_encode_frames',
           'cm_decode_frames', 'cm_encode_ex', 'cm_decode_ex', 'cm_encode_frames_host', 'cm_decode_frames_host',
           'cm_filter_rows', 'cm_transcode_frames_host', 'cm_measure_fma_peak', 'cm_launch_count', 'cm_timing_enable', 'cm_timing_reset', 'cm_timing_read', 'cm_phase_profile',
           'cm_yuv420p_to_rgb24', 'cm_rgb24_to_yuv420p', 'cm_encode_frames_host_fmt', 'cm_decode_frames_host_fmt',
           'cm_transcode_frames_host_fmt']

K_ENCODE, K_BANDSPLIT, K_PALD, K_COMB, K_DECODE_OTHER = 0, 1, 2, 3, 4

_lib = None


def load():
    """Load the shared library (once).  Raises NativeUnavailable with the reason if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeUnavailable('%s not built — run `python -c "import __graft_entry__ as g; g.build()"` '
                                '(there is no CPU fallback)' % LIB_PATH)
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:
        raise NativeUnavailable('cannot load %s: %s' % (LIB_PATH, e))
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.cm_abi_version.restype = C.c_int
    lib.cm_last_error.restype = C.c_char_p
    lib.cm_device_info.argtypes = [C.POINTER(C.c_int)] * 3
    lib.cm_create.argtypes = [C.POINTER(Desc), C.c_int, C.POINTER(vp)]
    lib.cm_destroy.argtypes = [vp]
    lib.cm_destroy.restype = None
    lib.cm_encode_frames.argtypes = [vp, vp, vp, i64, i32, vp]
    lib.cm_decode_frames.argtypes = [vp, vp, vp, i64, i32, vp]
    lib.cm_encode_ex.argtypes = [vp, C.POINTER(Window), vp, vp, vp, vp, i64, i32, vp]
    lib.cm_decode_ex.argtypes = [vp, C.POINTER(Window), vp, vp, vp, vp, i64, i32, vp]
    lib.cm_encode_frames_host.argtypes = [vp, vp, vp, i64, i32]
    lib.cm_decode_frames_host.argtypes = [vp, vp, vp, i64, i32]
    lib.cm_transcode_frames_host.argtypes = [vp, vp, vp, vp, i64, i32]
    pf = C.POINTER(PixFmt)
    lib.cm_yuv420p_to_rgb24.argtypes = [pf, vp, vp, i32, i32, i32, vp]
    lib.cm_rgb24_to_yuv420p.argtypes = [pf, vp, vp, i32, i32, i32, vp]
    lib.cm_encode_frames_host_fmt.argtypes = [vp, vp, vp, i64, i32, pf]
    lib.cm_decode_frames_host_fmt.argtypes = [vp, vp, vp, i64, i32, pf]
    lib.cm_transcode_frames_host_fmt.argtypes = [vp, vp, vp, vp, i64, i32, pf]
    lib.cm_measure_fma_peak.argtypes = [C.POINTER(C.c_double)]
    lib.cm_pald_matrix.argtypes = [vp, vp, C.POINTER(C.c_int)]
    lib.cm_filter_rows.argtypes = [C.POINTER(Filter), C.c_int, vp, vp, i32, vp]
    lib.cm_launch_count.restype = C.c_int64
    lib.cm_timing_enable.argtypes = [vp, C.c_int]
    lib.cm_timing_reset.argtypes = [vp]
    lib.cm_phase_profile.argtypes = [vp, vp]
    lib.cm_timing_read.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64)]
    if lib.cm_sizeof_desc() != C.sizeof(Desc):
        raise NativeUnavailable('cm_desc layout mismatch between %s and the Python binding' % LIB_NAME)
    if lib.cm_abi_version() != ABI_VERSION:
        raise NativeUnavailable('ABI version mismatch between %s and the Python binding' % LIB_NAME)
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise RuntimeError('color_modem_b200 native error %d: %s' % (rc, load().cm_last_error().decode()))


def launch_count():
    return int(load().cm_launch_count())
