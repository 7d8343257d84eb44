// Host-side internals shared by the translation units of libcolormodem_b200.so (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../../include/color_modem_b200.h"
#include "cm_common.cuh"

int cm_fail(int code, const char *fmt, const char *detail = "");
void cm_count_launch();

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) return cm_fail(CM_ERR_CUDA, #expr ": %s", cudaGetErrorString(_e)); \
    } while (0)

// Tuning knobs of a handle.  Read ONCE, in cm_create, from the environment (CM_ONEPASS, CM_ROWS_V1, CM_RPC, CM_CHUNK,
// CM_HOST_CHUNK, CM_ROWS_MAX, CM_MIN_WARPS, CM_OVERLAP, CM_PALD_MMA: A/B aids of tools/ab.py and of the alternative-path parity tests) — no launch
// path calls getenv.
struct cm_tune {
    bool onepass = false;      // legacy multi-row halo kernels instead of the two-pass row kernels
    bool rows_v1 = false;      // first-generation pass-1 kernel (k_qam_rows)
    int rpc = 0;               // rows a CTA of the row kernels walks through (the next one prefetched); 0 = cm_rows_per_cta decides
    int chunk = 0;             // frames per pass-1 / pass-2 launch pair (0: as many as a 2 GiB scratch holds)
    int host_chunk = 32;       // frames per host<->device chunk of the *_host entry points
    int host_roles = -1;       // 1: one stream per role (copy in / kernels / copy out), 4 buffers; 0: three streams, one chunk each;
                               // -1: by call — roles for encode->decode in one call (+8 %), streams for the single calls (two of which
                               // usually run side by side from two host threads: 24.4 k vs 22.0 k frames/s)
    int rows_max = 0;          // upper bound of rows per CTA of the multi-row kernels (0: none)
    int min_warps = 2;         // fewest warps per CTA of the multi-row kernels
    int mac_threads = 128;     // threads per CTA of the MAC kernels (CM_MAC_THREADS)
    bool pald_mma = true;      // PAL-D on the tensor cores where it serves the call (CM_PALD_MMA=0: the two-pass kernels)
    int overlap = 0;           // pass 2 of chunk i on a second stream under pass 1 of chunk i + 1 (measured: no gain, DESIGN.md section 5)
};

// PAL-D on the tensor cores (cm_pald_mma.cu): column tiles of TS output samples, N = 4 TS plane columns (a', b', LPpre a',
// LPpre b' of each sample), a K window of KW composite samples starting KPRE before the tile
#define CM_PALD_TS 32
#define CM_PALD_N (4 * CM_PALD_TS)
#define CM_PALD_KW 160
#define CM_PALD_KPRE 96

struct PaldMmaArgs {
    const uint16_t *b;      // [tile][hi | lo][KW / 8][N][8] FP16, the UMMA K-major layout without swizzle
    const float *cs;        // [tile][inverse column scale | bias][N]
    long long total;        // rows in the list of the call
    int per_frame;          // list rows per frame: len_a of the field of out_begin, then the other field's
    int len_a, row_a;       // rows listed for the field of out_begin, the first of them (the predecessor out_begin - 2)
    int nblocks;            // row tiles of 127 output lanes
};

struct cm_modem {
    cm_desc desc;
    cm_tune tune;
    int precision;
    int device;
    int sm_count;
    int smem_optin;
    DevParams<float> pf;
    DevParams<double> pd;
    MacConst<float> mcf;
    MacConst<double> mcd;
    void *d_tab = nullptr;
    void *d_taps = nullptr;
    void *d_ctab = nullptr;
    void *d_ptab = nullptr;
    void *d_mma_b = nullptr;    // PAL-D tensor-core kernel: B tiles and column scale / bias (plan_pald_mma); nullptr: not served
    void *d_mma_cs = nullptr;
    bool timing = false;
    unsigned long long *phase_prof = nullptr;
    // pairing scratch of the line-sequential decoders (grown on demand); one per host-path stream (+ slot 0 for
    // caller-provided streams: a handle must not be used from two streams at once)
    void *d_aux[12] = {};   // [which * 4 + slot]
    size_t aux_cap[12] = {};
    int aux_slot = 0;
    // two-pass decoders, device-resident calls: pass 2 (HBM-bound) of chunk i runs on s2 under pass 1 (issue-bound) of
    // chunk i + 1; ev_p1[b] = planes of buffer b written, ev_p2[b] = planes of buffer b consumed
    // a handle's scratch is shared by its device-resident calls: a call on another stream than the previous one first
    // waits for that one (event recorded after every call), so consecutive calls never race on the scratch
    cudaStream_t last_stream = nullptr;
    cudaEvent_t last_use = nullptr;
    bool used = false;
    cudaStream_t s2 = nullptr;
    cudaEvent_t ev_p1[2] = {nullptr, nullptr}, ev_p2[2] = {nullptr, nullptr};
    struct Ev { cudaEvent_t a, b; int id; };
    std::vector<Ev> events;
    // *_host entry points: the batch is cut into chunks that ping-pong over CM_HOST_STREAMS streams so that the
    // host->device copy of chunk i+1, the kernels of chunk i and the device->host copy of chunk i-1 overlap
    static const int kHostStreams = 3;          // by role: 0 host->device copies, 1 kernels, 2 device->host copies
    static const int kHostBufs = 4;             // staging buffers in flight
    cudaStream_t hs[kHostStreams] = {nullptr, nullptr, nullptr};
    void *d_in[kHostBufs] = {}, *d_out[kHostBufs] = {};
    void *d_mid[kHostBufs] = {};                // cm_transcode_frames_host: the composite between the two halves
    void *d_rgb[kHostBufs] = {};                // *_host_fmt with yuv420p: the RGB frames beside the link-side staging
    size_t in_cap[kHostBufs] = {}, out_cap[kHostBufs] = {}, mid_cap[kHostBufs] = {}, rgb_cap[kHostBufs] = {};
    cudaEvent_t ev_in[kHostBufs] = {}, ev_k[kHostBufs] = {}, ev_mid[kHostBufs] = {}, ev_out[kHostBufs] = {};
};

struct LaunchTimer {
    cm_modem *m;
    cudaStream_t st;
    cm_modem::Ev ev;
    bool on;
    LaunchTimer(cm_modem *m_, int id, cudaStream_t st_) : m(m_), st(st_), on(m_->timing) {
        if (on) {
            ev.id = id;
            cudaEventCreate(&ev.a);
            cudaEventCreate(&ev.b);
            cudaEventRecord(ev.a, st);
        }
    }
    ~LaunchTimer() {
        if (on) {
            cudaEventRecord(ev.b, st);
            m->events.push_back(ev);
        }
    }
};

// Rows per CTA of the one-row-at-a-time kernels: 2 for throughput (the next row's global load overlaps the current row),
// 1 when the launch is small (a single frame: twice the CTAs, half the latency — tools/latency.py).
static inline int cm_rows_per_cta(const cm_modem *m, long long rows_in_launch) {
    if (m->tune.rpc > 0) return m->tune.rpc;
    return rows_in_launch < 8LL * m->sm_count * 2 ? 1 : 2;
}

template <typename T> inline const DevParams<T> &params_of(const cm_modem *m);
template <> inline const DevParams<float> &params_of<float>(const cm_modem *m) { return m->pf; }
template <> inline const DevParams<double> &params_of<double>(const cm_modem *m) { return m->pd; }

template <typename K>
static int set_smem(K kernel, size_t bytes) {
    CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return CM_OK;
}

// Largest R in [1, rmax] whose shared-memory footprint fits `budget`; 0 if even R = 1 does not fit.
// cm_tune::rows_max lowers rmax.
template <class F>
static int pick_rows(const cm_modem *m, int rmax, size_t budget, F bytes_for) {
    if (m->tune.rows_max >= 1 && m->tune.rows_max < rmax) rmax = m->tune.rows_max;
    for (int r = rmax; r >= 1; --r)
        if (bytes_for(r) <= budget) return r;
    return 0;
}

// Threads per CTA for `tasks` concurrent warp-level IIR tasks: one warp per task, at least two.  Small CTAs win on
// B200 for these kernels (measured sweep of rows per CTA x warps, DESIGN.md section 5): many independent CTAs per SM
// in different phases overlap better than a few large ones that synchronise 8 warps at every phase boundary.
static inline int cta_threads(const cm_modem *m, int tasks) {
    const int minw = m->tune.min_warps;
    int warps = tasks < minw ? minw : tasks;
    if (warps > CM_NWARPS) warps = CM_NWARPS;
    return 32 * warps;
}

template <typename T>
static void set_groups(IoArgs<T> &io, int R) {
    io.rows_per_cta = R;
    int rows_in_field = (io.out_count + 1) >> 1;
    io.groups_per_field = (rows_in_field + R - 1) / R;
}

// grid of a row-group kernel: x = groups per field, y = 2 fields, z = frames (run_ex keeps nframes <= 65535 per launch)
template <typename T>
static dim3 cm_grid(const IoArgs<T> &io) {
    return dim3((unsigned)io.groups_per_field, 2u, (unsigned)io.nframes);
}

// rows of [begin, begin+count) that have no predecessor in the window (r < 2) / that have one (r >= 2)
template <typename T>
static void split_top(const IoArgs<T> &io, IoArgs<T> &top, IoArgs<T> &rest) {
    top = io;
    rest = io;
    int end = io.out_begin + io.out_count;
    int top_end = end < 2 ? end : 2;
    top.out_count = top_end > io.out_begin ? top_end - io.out_begin : 0;
    int rest_begin = io.out_begin > 2 ? io.out_begin : 2;
    rest.out_begin = rest_begin;
    rest.out_count = end > rest_begin ? end - rest_begin : 0;
}

// Grow-only device scratch of a handle (stream-ordered use only).
// which = 0: pass-1 -> pass-2 planes; 1: (y, u, v) rows waiting for the luma notch; 2: second planes buffer (overlap)
void *cm_ensure_aux(cm_modem *m, size_t bytes, int which = 0);   // nullptr on failure (cm_last_error set)

// Explicit instantiation of the float / double variants; the build may compile a unit once per type
// (-DCM_INST_F32 / -DCM_INST_F64) so that the two halves compile in parallel.
#if defined(CM_INST_F32)
#define CM_INSTANTIATE(f32, f64) f32
#elif defined(CM_INST_F64)
#define CM_INSTANTIATE(f32, f64) f64
#else
#define CM_INSTANTIATE(f32, f64) f32 f64
#endif

// per-family entry points (explicitly instantiated for float and double in cm_<family>.cu)
template <typename T> int qam_encode(cm_modem *m, IoArgs<T> io, cudaStream_t st);
template <typename T> int qam_decode(cm_modem *m, IoArgs<T> io, int mode, cudaStream_t st);
template <typename T> int secam_encode(cm_modem *m, IoArgs<T> io, cudaStream_t st);
template <typename T> int secam_decode(cm_modem *m, IoArgs<T> io, cudaStream_t st);
template <typename T> int niir_encode(cm_modem *m, IoArgs<T> io, cudaStream_t st);
template <typename T> int niir_decode(cm_modem *m, IoArgs<T> io, cudaStream_t st);
template <typename T> int proto_encode(cm_modem *m, IoArgs<T> io, cudaStream_t st);
template <typename T> int proto_decode(cm_modem *m, IoArgs<T> io, cudaStream_t st);
template <typename T> int mac_encode(cm_modem *m, IoArgs<T> io, cudaStream_t st);
template <typename T> int mac_decode(cm_modem *m, IoArgs<T> io, cudaStream_t st);
int launch_pald_mma(cm_modem *m, IoArgs<float> io, cudaStream_t st);
