/*
 * color_modem_b200 — C ABI of the B200-native colour-modem hot path.
 *
 * The reference (kFYatek/color_modem) is pure Python and has no FFI; its boundary is the duck-typed modem
 * protocol (SURVEY.md §8b).  This header is what a binding for that protocol would call:
 *
 *   reference interface                                            replaced by
 *   ---------------------------------------------------------------------------------------------------
 *   modem constructors (color/ntsc.py:24,53  color/pal.py:29,63,131    cm_create()  — the host keeps doing the
 *     color/secam.py:153  color/niir.py:11,167  color/protosecam.py:29   scipy filter *design* (utils.py:39-64) and
 *     color/mac.py:16  comb.py:72,126,131)                              hands the coefficients over in cm_desc
 *   ImageModem.modulate(img, frame)        image.py:27-56           cm_encode_frames()
 *   ImageModem.demodulate(img, frame)      image.py:58-84           cm_decode_frames()
 *   modem.modulate(frame, line, r, g, b)   qam.py:68-69 etc.        cm_encode_ex() on a 1..3-row window
 *   modem.demodulate(frame, line, comp)    qam.py:71-72 etc.        cm_decode_ex() on a 1..5-row window
 *                                                                    (see cm_window below)
 *   modem.modulate_components / demodulate_components               the same two calls on a handle created with identity
 *     ntsc.py:43-49  pal.py:48-59,180-234  comb.py:40-59             colour matrices (planes in, planes out)
 *     niir.py:80,98  secam.py:261  protosecam.py:74  mac.py:42
 *   QamColorModem.modulate / demodulate / extract_chroma            cm_encode_ex / cm_decode_ex with cm_window.phase_offset
 *     qam.py:28-58                                                   (explicit start phase), CM_MODE_EXTRACT_CHROMA
 *   FilterFunction.__call__                utils.py:28-36           cm_filter_rows()
 *
 * Conventions: every function returns 0 on success or a negative cm_status; it never throws.  All frame
 * pointers are DEVICE pointers owned by the caller (cm_*_host variants take HOST pointers and do the copies
 * themselves).  `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  A handle is bound
 * to the CUDA device that was current in cm_create and is not re-entrant.
 */
#ifndef COLOR_MODEM_B200_H
#define COLOR_MODEM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CM_ABI_VERSION 3

enum cm_status {
    CM_OK = 0,
    CM_ERR_INVALID = -1,      /* bad descriptor / argument */
    CM_ERR_CUDA = -2,         /* CUDA runtime error, see cm_last_error() */
    CM_ERR_UNSUPPORTED = -3,  /* composition not built */
    CM_ERR_NOMEM = -4
};

/* Modem composition (which reference class stack the handle stands for). */
enum cm_kind {
    CM_KIND_QAM_BANDSPLIT = 1, /* NtscModem (ntsc.py:23-49) / PalSModem (pal.py:28-59)                  */
    CM_KIND_NTSC_COMB = 2,     /* NtscCombModem (ntsc.py:52-82)                                         */
    CM_KIND_NTSC_3D = 3,       /* Simple3DCombModem(NtscCombModem) (comb.py:71-127)                      */
    CM_KIND_PAL_D = 4,         /* PalDModem (pal.py:62-127)                                             */
    CM_KIND_PAL_3D = 5,        /* Pal3DModem (pal.py:130-234)                                           */
    CM_KIND_SECAM = 6,         /* SecamModem (secam.py:152-304)                                         */
    CM_KIND_NIIR = 7,          /* NiirModem / HueCorrectingNiirModem (niir.py)                           */
    CM_KIND_PROTOSECAM = 8,    /* ProtoSecamModem (protosecam.py:28-112)                                 */
    CM_KIND_MAC = 9            /* MacModem (mac.py:15-125)                                              */
};

enum cm_flags {
    CM_FLAG_PAL_VSWITCH = 1,   /* V sign alternates line by line (pal.py:48-59)                          */
    CM_FLAG_CHROMA_AVG = 2,    /* encoder wrapped in ColorAveragingModem (comb.py:130-167)               */
    CM_FLAG_HUE_CORRECT = 4,   /* HueCorrectingNiirModem encoder (niir.py:166-202)                       */
    CM_FLAG_NTSC_NO_COMB = 8,  /* NtscCombModem with |sin(LS/2)| <= 0.05: falls back to band-split chroma */
    CM_FLAG_PAL3D_SIN = 16,    /* Pal3DModem use_sin (pal.py:155-165)                                    */
    CM_FLAG_PAL3D_COS = 32,    /* Pal3DModem use_cos                                                     */
    CM_FLAG_SECAM_BELL = 64,   /* SECAM anti-bell filter present (secam.py:167-170)                      */
    CM_FLAG_SECAM_LF = 128,    /* SECAM LF pre-/de-emphasis present (secam.py:173-177)                   */
    CM_FLAG_PROTO_LUMA = 256,  /* ProtoSecam premod_luma_filter (protosecam.py:82-85)                    */
    CM_FLAG_NOTCH = 512,       /* comb decoders: luma notch after the chroma subtraction (comb.py:18-20,54-55) */
    CM_FLAG_MINAVG = 1024      /* 3-line decoders: avg=comb.minavg instead of the mean (comb.py:13-15, pal.py:146-149) */
};

enum cm_precision { CM_FP32 = 0, CM_FP64 = 1 };

#define CM_MAX_SECTIONS 6
#define CM_MAX_FILTERS 10
#define CM_MAX_SCALARS 48
#define CM_MAX_RESAMPLERS 6
#define CM_MAX_TAPS 1024

/* One IIR use-site: FilterFunction (utils.py:9-36) as a cascade of biquads  (b0 b1 b2 a1 a2, a0 = 1),
 * designed on the host by the same scipy calls as the reference and converted to second-order sections in
 * float64.  `shift` is the integer group-delay compensation of utils.py:19-22 (edge-replicate tail). */
typedef struct cm_filter {
    int32_t nsec;
    int32_t shift;
    int32_t n;        /* input length at this use-site (samples per line at the rate the filter runs at) */
    int32_t rate;     /* 1, 2 or 3: oversampling factor the filter runs at (selects the shared-memory layout) */
    double sos[CM_MAX_SECTIONS][5];
} cm_filter;

/* One resample_poly use-site (qam.py:35 etc.): out[j] = sum_i x[i] * taps[half + j*down - i*up]. */
typedef struct cm_resampler {
    int32_t up, down, half, ntaps;
    double taps[CM_MAX_TAPS];
} cm_resampler;

/* Everything a handle needs.  Slot meanings of filters[]/scalars[]/phases[] are per kind and are documented
 * next to the kernels (color_modem_b200/csrc/cm_slots.h); the Python host fills them (color_modem_b200/*.py). */
typedef struct cm_desc {
    int32_t abi_version;      /* CM_ABI_VERSION */
    int32_t kind;             /* cm_kind */
    int32_t flags;            /* cm_flags */
    int32_t width, height;    /* RGB raster */
    int32_t comp_width;       /* composite samples per line (== width except MAC) */
    int32_t out_width;        /* decoded RGB samples per line (== width except MAC: 720) */
    /* raster (line.py:50-65) */
    int32_t digital_shift;    /* LineConfig._line_shift */
    int32_t odd_first, even_first, ref_line;
    int32_t frame_cycle;      /* utils.py:78-80 */
    /* subcarrier phase, in turns as 0.64 fixed point (wraps mod 1 turn == mod 2*pi) */
    uint64_t frame_shift_turns;   /* frac(fsc / frame_rate)                utils.py:74-76 */
    uint64_t line_shift_turns;    /* frac(fsc / (frame_rate*total_lines))  utils.py:69-72 */
    uint64_t phases[16];          /* per-kind constant phase offsets / per-sample steps, in turns */
    double scalars[CM_MAX_SCALARS];
    double enc_matrix[9];     /* rows: (y, c1, c2) from (r, g, b)   e.g. ntsc.py:28-33 */
    double dec_matrix[9];     /* rows: (r, g, b)  from (y, c1, c2)  e.g. ntsc.py:36-41 */
    int32_t nfilters;
    cm_filter filters[CM_MAX_FILTERS];
    int32_t nresamplers;
    cm_resampler resamplers[CM_MAX_RESAMPLERS];
} cm_desc;

typedef struct cm_modem cm_modem;

/* Row window.  A launch works on buffers holding `nrows` consecutive raster rows per frame; buffer row r is
 * line number y0 + r, rows r-2 / r+2 are its same-field neighbours, and a row without a predecessor in the
 * buffer behaves as the top of its field (the reference's "line != last_line + 2" reset, e.g. comb.py:48), a
 * row without a successor as the bottom of its field (image.py:51-53 re-feeds the row itself).  Only rows
 * [out_begin, out_begin + out_count) are computed.  Whole frames are the window {height, 0, 0, height}; the
 * per-line protocol (modem.modulate / modem.demodulate, qam.py:68-72) uses 1..5-row windows. */
typedef struct cm_window {
    int32_t nrows;
    int32_t y0;
    int32_t out_begin;
    int32_t out_count;
    int32_t mode;       /* cm_window_mode; 0 for the composition's normal behaviour */
    int32_t reserved;
    uint64_t phase_offset;  /* added to the subcarrier phase at the first sample of every row, in turns as 0.64 fixed
                             * point.  With a descriptor whose frame / line shifts are zero this is the explicit
                             * start_phase argument of QamColorModem.modulate / demodulate (qam.py:28,43); 0 otherwise */
} cm_window;

enum cm_window_mode {
    CM_MODE_DEFAULT = 0,
    /* decode: what backend.demodulate_components(..., strip_chroma=False) returns — band-split chroma with the
     * composite itself as luma.  This is the value the stateful comb decoders hand back from their reset branch
     * (pal.py:191-195, comb.py:97-99); ImageModem discards it, the per-line protocol exposes it. */
    CM_MODE_BANDSPLIT_NOSTRIP = 1,
    /* decode, QAM family: QamColorModem.extract_chroma (qam.py:34-37), down2(BP(up2 composite)), returned in the first
     * output plane (the other two are zero) */
    CM_MODE_EXTRACT_CHROMA = 2
};

int cm_abi_version(void);
/* sizeof(cm_desc) as compiled into the library (lets a foreign-language binding verify its struct layout). */
int cm_sizeof_desc(void);
const char *cm_last_error(void);
int cm_device_info(int *sm_count, int *cc_major, int *cc_minor);

/* Line widths (width, comp_width, out_width) must be multiples of 4 samples, u8 frame pointers 4-byte aligned and float
 * frame pointers 16-byte (float) / 8-byte (double) aligned: the kernels move four samples per 32-bit / 96-bit / 128-bit
 * access (a float vector of four samples in one access).  cm_encode_ex / cm_decode_ex refuse a misaligned frame pointer
 * with CM_ERR_INVALID before any launch.  (The reference accepts any width: image.py:27-84.)  The tuning knobs of a handle
 * are read from the environment here, once. */
int cm_create(const cm_desc *desc, int precision, cm_modem **out);
void cm_destroy(cm_modem *m);

/* ImageModem.modulate over a batch (image.py:27-56): rgb u8 [n][H][W][3] -> comp u8 [n][H][Wc].
 * Frame i of the batch is absolute frame first_frame + i (carrier phase and line parity depend on it). */
int cm_encode_frames(cm_modem *m, const uint8_t *rgb, uint8_t *comp, int64_t first_frame, int32_t nframes,
                     void *stream);

/* ImageModem.demodulate over a batch (image.py:58-84): comp u8 [n][H][Wc] -> rgb u8 [n][H][Wo][3]. */
int cm_decode_frames(cm_modem *m, const uint8_t *comp, uint8_t *rgb, int64_t first_frame, int32_t nframes,
                     void *stream);

/* General form.  win == NULL means whole frames.  Exactly one of the inputs must be non-NULL, at least one of
 * the outputs.  Float buffers are of the handle's precision (float or double):
 *   rgb_float  [n][nrows][W][3]   RGB in [0,1] as handed to modem.modulate
 *   comp_float [n][nrows][Wc]     composite as returned by modem.modulate (BEFORE the 0.6v+0.2 level map) /
 *                                 as handed to modem.demodulate (AFTER the (5v-1)/3 un-level map)
 *   rgb_float out [n][nrows][Wo][3]  as returned by modem.demodulate (before clipping). */
int cm_encode_ex(cm_modem *m, const cm_window *win, const uint8_t *rgb_u8, const void *rgb_float,
                 uint8_t *comp_u8, void *comp_float, int64_t first_frame, int32_t nframes, void *stream);
int cm_decode_ex(cm_modem *m, const cm_window *win, const uint8_t *comp_u8, const void *comp_float,
                 uint8_t *rgb_u8, void *rgb_float, int64_t first_frame, int32_t nframes, void *stream);

/* Whole frames with HOST buffers: copies in, runs, copies out, synchronises. */
int cm_encode_frames_host(cm_modem *m, const uint8_t *rgb, uint8_t *comp, int64_t first_frame, int32_t nframes);
int cm_decode_frames_host(cm_modem *m, const uint8_t *comp, uint8_t *rgb, int64_t first_frame, int32_t nframes);

/* ImageModem.modulate followed by ImageModem.demodulate of the result (the sequence of the reference's cli.py:62-65) in
 * one call with HOST buffers: rgb_in [n][H][W][3] -> rgb_out [n][H][Wo][3].  The composite stays in device memory between
 * the two halves; it is copied out to comp_out [n][H][Wc] as well unless comp_out is NULL.  Same bytes as the two calls
 * above, one host->device trip less. */
int cm_transcode_frames_host(cm_modem *m, const uint8_t *rgb_in, uint8_t *comp_out, uint8_t *rgb_out, int64_t first_frame,
                             int32_t nframes);

/* Picture format of the frame-batch paths.  CM_PIX_RGB24: packed [H][W][3] bytes, the format of every call above.
 * CM_PIX_YUV420P: planar 8-bit YUV 4:2:0 (I420): Y [H][W], then U (Cb) [ceil(H/2)][W/2], then V (Cr) [ceil(H/2)][W/2];
 * W * H + 2 * (W/2) * ceil(H/2) bytes per frame; chroma rows are 2-byte aligned only.  `matrix` and `range` select the
 * colour matrix (BT.601: Kr 0.299, Kb 0.114; BT.709: Kr 0.2126, Kb 0.0722) and the quantisation (limited: Y' 16..235,
 * C 16..240; full: 0..255).  The conversion is exact integer arithmetic in Q16 (INTEGRATION.md, "Picture formats"):
 * RGB -> YUV averages each 2x2 chroma block (an odd height's last row counts twice), YUV -> RGB upsamples the chroma by
 * nearest neighbour.  `reserved` must be 0. */
enum cm_pix_format { CM_PIX_RGB24 = 0, CM_PIX_YUV420P = 1 };
enum cm_yuv_matrix { CM_YUV_BT601 = 0, CM_YUV_BT709 = 1 };
enum cm_yuv_range { CM_YUV_LIMITED = 0, CM_YUV_FULL = 1 };
typedef struct cm_pixfmt {
    int32_t format, matrix, range, reserved;
} cm_pixfmt;

/* Device conversions between yuv420p [n][frame bytes] and rgb24 [n][H][W][3] (DEVICE pointers).  f->format must be
 * CM_PIX_YUV420P; width a multiple of 4.  Stream-ordered, allocate nothing, may be captured in a CUDA graph. */
int cm_yuv420p_to_rgb24(const cm_pixfmt *f, const uint8_t *yuv, uint8_t *rgb, int32_t width, int32_t height, int32_t nframes,
                        void *stream);
int cm_rgb24_to_yuv420p(const cm_pixfmt *f, const uint8_t *rgb, uint8_t *yuv, int32_t width, int32_t height, int32_t nframes,
                        void *stream);

/* The three HOST-buffer calls above with the picture side in format `f` (f == NULL or CM_PIX_RGB24: exactly the calls
 * above).  For CM_PIX_YUV420P the picture buffers hold yuv420p frames: W wide on the input side, Wo wide on the output side;
 * only those bytes cross the link, the conversions run on the device before the encoder and after the decoder. */
int cm_encode_frames_host_fmt(cm_modem *m, const uint8_t *pic, uint8_t *comp, int64_t first_frame, int32_t nframes,
                              const cm_pixfmt *f);
int cm_decode_frames_host_fmt(cm_modem *m, const uint8_t *comp, uint8_t *pic, int64_t first_frame, int32_t nframes,
                              const cm_pixfmt *f);
int cm_transcode_frames_host_fmt(cm_modem *m, const uint8_t *pic_in, uint8_t *comp_out, uint8_t *pic_out,
                                 int64_t first_frame, int32_t nframes, const cm_pixfmt *f);

/* FilterFunction.__call__ (utils.py:28-36) on `nrows` independent rows of f->n samples each: causal IIR from zero
 * state, the input extended by f->shift copies of its last sample and the first f->shift outputs dropped.  `in` / `out`
 * are DEVICE buffers [nrows][f->n] of the given precision (float or double); f->rate is ignored.  Synchronises the
 * stream.  Carrier of the reference's L0 filter kit and of the luma notch of composed comb wrappers (comb.py:18-20). */
int cm_filter_rows(const cm_filter *f, int precision, const void *in, void *out, int32_t nrows, void *stream);

/* Optional per-kernel device timing (CUDA events recorded on the launch stream around every kernel launch).
 * bench.py uses it for the roofline line; it is off by default and costs nothing when off. */
enum cm_kernel_id {
    CM_K_ENCODE = 0,       /* fused encode kernel of the handle's family */
    CM_K_BANDSPLIT = 1,    /* k_qam_bandsplit */
    CM_K_PALD = 2,         /* k_pald_combed */
    CM_K_COMB = 3,         /* k_qam_comb */
    CM_K_DECODE_OTHER = 4, /* decode kernels of the non-QAM families */
    CM_K_COUNT = 5
};
int cm_timing_enable(cm_modem *m, int on);
int cm_timing_reset(cm_modem *m);
/* Waits for the recorded events; returns summed milliseconds and number of launches of kernel `id`. */
int cm_timing_read(cm_modem *m, int id, double *total_ms, int64_t *launches);

/* Tuning aid: when `device_counters` (>= 32 zeroed uint64 on the device) is non-NULL, instrumented kernels add the
 * cycles thread 0 of every CTA spends between consecutive barriers to counters[phase].  NULL switches it off. */
int cm_phase_profile(cm_modem *m, void *device_counters);

/* Measured FP32 multiply-add peak of the current device in 1e12 multiply-adds per second (packed FFMA2 with uniform
 * operands, every SM full): the denominator of bench.py's roofline_fma.  Takes ~20 ms. */
int cm_measure_fma_peak(double *tfma_per_s);

/* Number of kernel launches issued by this library in the calling process (bench.py's gpu_launches). */
int64_t cm_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif
