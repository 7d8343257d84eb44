// Launchers of the QAM family (NTSC / PAL): kernels in cm_qam.cuh.
//
// The build compiles this file several times (__graft_entry__.py: UNIT_VARIANTS): -DCM_QAM_PART=0 encoder and
// band-split kernels, 1 PAL-D kernel, 2 line-comb kernels, 3 the dispatchers; -DCM_INST_F32 / -DCM_INST_F64 keep one
// arithmetic type.  Without the macros everything lands in one object.
#include "cm_host.h"
#include "cm_qam.cuh"

#ifdef CM_QAM_PART
#define CM_PART(n) (CM_QAM_PART == (n))
#else
#define CM_PART(n) 1
#endif

template <typename T> int launch_bandsplit(cm_modem *m, IoArgs<T> io, int luma_mode, cudaStream_t st);
template <typename T> int launch_pald(cm_modem *m, IoArgs<T> io, cudaStream_t st);
template <typename T> int launch_extract(cm_modem *m, IoArgs<T> io, cudaStream_t st);
template <typename T, int MODE> int launch_comb(cm_modem *m, IoArgs<T> io, cudaStream_t st);
template <typename T> int qam_decode(cm_modem *m, IoArgs<T> io, int mode, cudaStream_t st);

// true when some IIR use-site of the handle spans several super-chunks (long lines): use the multi-warp kernels
template <typename T>
static bool needs_teams(const DevParams<T> &p) {
    for (int i = 0; i < CM_NFILT; ++i)
        if (p.filt[i].nsec && p.filt[i].nsuper > 1) return true;
    return false;
}

// threads of a one-row CTA: two concurrent IIR tasks, each run by a team of `nsuper` warps (at most 4, cm_iir.cuh)
template <typename T>
static int row_threads(const DevParams<T> &p) {
    int ts = 1;
    for (int i = 0; i < CM_NFILT; ++i)
        if (p.filt[i].nsec && p.filt[i].nsuper > ts) ts = p.filt[i].nsuper;
    if (ts > 4) ts = 1;
    return 64 * ts;
}

#if CM_PART(0)
template <typename T>
int qam_encode(cm_modem *m, IoArgs<T> io, cudaStream_t st) {
    const DevParams<T> &p = params_of<T>(m);
    if (io.out_count <= 0) return CM_OK;
    auto bytes = [&](int r) { return (128 + (size_t)r * 3 * p.n1p) * sizeof(T); };
    int R = pick_rows(m, 1, (size_t)m->smem_optin / 2, bytes);     // one row, two warps (u and v low-pass): 1.84 vs 2.64 us/frame
    if (!R) return cm_fail(CM_ERR_UNSUPPORTED, "line too wide for the encode kernel%s");
    const bool teams = needs_teams(p);
    if (io.in_u8 && p.enc_geo && !m->tune.onepass && !m->tune.rows_v1) {     // second-generation row encoder
        void (*kern)(const DevParams<T>, const IoArgs<T>) =
            p.enc_geo == 1 ? k_qam_encode_row2<T, 1> : (p.enc_geo == 2 ? k_qam_encode_row2<T, 2> : k_qam_encode_row2<T, 3>);
        int rc1 = set_smem(kern, bytes(1));
        if (rc1) return rc1;
        const int rpc = cm_rows_per_cta(m, (long long)io.out_count * io.nframes);
        const int nf = (io.out_count + 1) >> 1;
        {
            LaunchTimer lt(m, CM_K_ENCODE, st);
            kern<<<dim3((unsigned)((nf + rpc - 1) / rpc), 2u, (unsigned)io.nframes), p.enc_geo == 1 ? 64 : 128, bytes(1), st>>>(p, io);
        }
        cm_count_launch();
        CUDA_TRY(cudaGetLastError());
        return CM_OK;
    }
    if (!teams && io.in_u8 && p.W <= 768 && !m->tune.onepass) {        // one row at a time, next row prefetched
        int rc1 = set_smem(k_qam_encode_row<T>, bytes(1));
        if (rc1) return rc1;
        const int rpc = cm_rows_per_cta(m, (long long)io.out_count * io.nframes);
        const int nf = (io.out_count + 1) >> 1;
        {
            LaunchTimer lt(m, CM_K_ENCODE, st);
            k_qam_encode_row<T><<<dim3((unsigned)((nf + rpc - 1) / rpc), 2u, (unsigned)io.nframes), CM_ROW_THREADS, bytes(1), st>>>(p, io);
        }
        cm_count_launch();
        CUDA_TRY(cudaGetLastError());
        return CM_OK;
    }
    set_groups(io, R);
    int rc = teams ? set_smem(k_qam_encode<T, true>, bytes(R)) : set_smem(k_qam_encode<T, false>, bytes(R));
    if (rc) return rc;
    dim3 grid = cm_grid(io);
    {
        LaunchTimer lt(m, CM_K_ENCODE, st);
        if (teams) k_qam_encode<T, true><<<grid, CM_NTHREADS, bytes(R), st>>>(p, io);
        else k_qam_encode<T, false><<<grid, cta_threads(m, 2 * R), bytes(R), st>>>(p, io);
    }
    cm_count_launch();
    CUDA_TRY(cudaGetLastError());
    return CM_OK;
}

template <typename T>
int launch_bandsplit(cm_modem *m, IoArgs<T> io, int luma_mode, cudaStream_t st) {
    const DevParams<T> &p = params_of<T>(m);
    if (io.out_count <= 0) return CM_OK;
    auto bytes = [&](int r) { return (CM_TAPS_ELEMS + (size_t)r * (p.n1p + 8 * (size_t)p.hb2)) * sizeof(T); };
    int R = pick_rows(m, 4, (size_t)m->smem_optin / 2, bytes);
    if (!R) R = pick_rows(m, 1, (size_t)m->smem_optin, bytes);
    if (!R) return cm_fail(CM_ERR_UNSUPPORTED, "line too wide for the band-split kernel%s");
    const bool teams = needs_teams(p);
    if (luma_mode == 0 && p.kind == CM_KIND_QAM_BANDSPLIT && p.row_geo && !m->tune.onepass && !m->tune.rows_v1) {
        const size_t b2 = (128 + (size_t)p.n1p + 6 * (size_t)p.hb2) * sizeof(T);
        if (b2 <= (size_t)m->smem_optin) {
            void (*kern)(const DevParams<T>, const IoArgs<T>) =
                p.row_geo == 1 ? k_qam_bs_row2<T, 1> : (p.row_geo == 2 ? k_qam_bs_row2<T, 2> : k_qam_bs_row2<T, 3>);
            int rc2 = set_smem(kern, b2);
            if (rc2) return rc2;
            const int rpc = cm_rows_per_cta(m, (long long)io.out_count * io.nframes);
            {
                LaunchTimer lt(m, CM_K_BANDSPLIT, st);
                kern<<<dim3((unsigned)((io.out_count + rpc - 1) / rpc), 1u, (unsigned)io.nframes), p.row_geo == 1 ? 64 : 128, b2, st>>>(p, io);
            }
            cm_count_launch();
            CUDA_TRY(cudaGetLastError());
            return CM_OK;
        }
    }
    if (luma_mode == 0 && !m->tune.onepass) {       // one row per CTA: two IIR tasks, one warp (team) each
        const size_t b1 = (128 + (size_t)p.n1p + 8 * (size_t)p.hb2) * sizeof(T);
        if (b1 <= (size_t)m->smem_optin) {
            int rc1 = teams ? set_smem(k_qam_bs_row<T, true>, b1) : set_smem(k_qam_bs_row<T, false>, b1);
            if (rc1) return rc1;
            const dim3 grid((unsigned)io.out_count, 1u, (unsigned)io.nframes);
            {
                LaunchTimer lt(m, CM_K_BANDSPLIT, st);
                if (teams) k_qam_bs_row<T, true><<<grid, row_threads(p), b1, st>>>(p, io);
                else k_qam_bs_row<T, false><<<grid, CM_ROW_THREADS, b1, st>>>(p, io);
            }
            cm_count_launch();
            CUDA_TRY(cudaGetLastError());
            return CM_OK;
        }
    }
    set_groups(io, R);
    int rc = teams ? set_smem(k_qam_bandsplit<T, true>, bytes(R)) : set_smem(k_qam_bandsplit<T, false>, bytes(R));
    if (rc) return rc;
    dim3 grid = cm_grid(io);
    {
        LaunchTimer lt(m, CM_K_BANDSPLIT, st);
        if (teams) k_qam_bandsplit<T, true><<<grid, CM_NTHREADS, bytes(R), st>>>(p, io, luma_mode);
        else k_qam_bandsplit<T, false><<<grid, cta_threads(m, 2 * R), bytes(R), st>>>(p, io, luma_mode);
    }
    cm_count_launch();
    CUDA_TRY(cudaGetLastError());
    return CM_OK;
}

template <typename T>
int launch_extract(cm_modem *m, IoArgs<T> io, cudaStream_t st) {
    const DevParams<T> &p = params_of<T>(m);
    if (io.out_count <= 0) return CM_OK;
    if (!io.out_f) return cm_fail(CM_ERR_INVALID, "CM_MODE_EXTRACT_CHROMA needs a float output buffer%s");
    const size_t b1 = (128 + (size_t)p.n1p + 2 * (size_t)p.hb2) * sizeof(T);
    if (b1 > (size_t)m->smem_optin) return cm_fail(CM_ERR_UNSUPPORTED, "line too wide for the extract kernel%s");
    int rc = set_smem(k_qam_extract<T>, b1);
    if (rc) return rc;
    k_qam_extract<T><<<dim3((unsigned)io.out_count, 1u, (unsigned)io.nframes), CM_NTHREADS, b1, st>>>(p, io);
    cm_count_launch();
    CUDA_TRY(cudaGetLastError());
    return CM_OK;
}

CM_INSTANTIATE(template int launch_extract<float>(cm_modem *, IoArgs<float>, cudaStream_t);,
               template int launch_extract<double>(cm_modem *, IoArgs<double>, cudaStream_t);)
CM_INSTANTIATE(template int qam_encode<float>(cm_modem *, IoArgs<float>, cudaStream_t);,
               template int qam_encode<double>(cm_modem *, IoArgs<double>, cudaStream_t);)
CM_INSTANTIATE(template int launch_bandsplit<float>(cm_modem *, IoArgs<float>, int, cudaStream_t);,
               template int launch_bandsplit<double>(cm_modem *, IoArgs<double>, int, cudaStream_t);)
#endif

#if CM_PART(1) || CM_PART(2)
// Two-pass decoders over independent rows (cm_qam.cuh: k_qam_rows<PALD / STD>, then k_qam_combine<MODE>).  The batch
// is cut into chunks whose plane scratch (16 B per pixel) stays within 2 GiB.
template <typename T, int MODE>
int launch_rows_pair(cm_modem *m, IoArgs<T> io, cudaStream_t st) {
    const DevParams<T> &p = params_of<T>(m);
    if (io.out_count <= 0) return CM_OK;
    if constexpr (MODE == PAIR_PALD && IsF32<T>::value) {
        // u8 composite (exact in FP16) without the (y, u, v) diversion of the non-default knobs: one kernel on the
        // tensor cores when the handle has its band matrix (cm_api.cu: plan_pald_mma)
        if (m->d_mma_b && io.in_u8 && !io.yuv) return launch_pald_mma(m, io, st);
    }
    size_t b1 = (128 + (size_t)p.n1p + 6 * (size_t)p.hb2) * sizeof(T);
    const bool teams = needs_teams(p);
    constexpr bool kPald = MODE == PAIR_PALD;
    void (*pass1)(const DevParams<T>, const IoArgs<T>) = teams ? k_qam_rows<T, kPald, true> : k_qam_rows<T, kPald, false>;
    int threads1 = teams ? row_threads(p) : CM_ROW_THREADS;
    if (p.row_geo && !m->tune.rows_v1) {
        pass1 = p.row_geo == 1 ? k_qam_rows2<T, kPald, 1> : (p.row_geo == 2 ? k_qam_rows2<T, kPald, 2> : k_qam_rows2<T, kPald, 3>);
        threads1 = p.row_geo == 1 ? 64 : 128;
        b1 = (128 + 2 * (size_t)p.n1p + 4 * (size_t)p.hb2) * sizeof(T);
    }
    if (b1 > (size_t)m->smem_optin) return cm_fail(CM_ERR_UNSUPPORTED, "line too wide for the row kernels%s");
    int rc = set_smem(pass1, b1);
    if (rc) return rc;
    // Frames per pass-1 / pass-2 launch pair.  Pass 1 is bound by instruction issue, pass 2 by HBM: with the batch cut into
    // chunks, pass 2 of chunk i runs on a second (high-priority) stream while pass 1 of chunk i + 1 runs on the caller's,
    // the planes double-buffered (cm_tune::overlap; device-resident calls only — the host entry points already pipeline
    // their chunks over three streams).  Without overlap a chunk is as large as a 2 GiB scratch allows (720x576: 6.6 MB
    // per frame -> 323 frames; 1920x1080: 33 MB -> 64): measured on 256 PAL-D frames, serial, 32 per launch 81.7 k,
    // 64: 86.5 k, 128: 88.8 k, 256: 89.9 k frames/s.
    const size_t frame_elems = (size_t)io.nrows * 4 * p.W;
    int kChunk = (int)(((size_t)2 << 30) / (frame_elems * sizeof(T)));
    if (kChunk < 16) kChunk = 16;
    bool overlap = m->tune.overlap && m->aux_slot == 0;
    if (overlap) {
        // chunks of ~1/4 of the batch, at least 32 frames of 720x576 worth of rows: enough CTAs per launch to fill the chip
        int c = (io.nframes + 3) / 4;
        const int min_frames = (int)((32ull * 576 * 720 + (size_t)io.nrows * p.W - 1) / ((size_t)io.nrows * p.W));
        if (c < min_frames) c = min_frames;
        if (c < kChunk) kChunk = c;
    }
    if (m->tune.chunk > 0) kChunk = m->tune.chunk;
    const int chunk = io.nframes < kChunk ? io.nframes : kChunk;
    if (chunk >= io.nframes) overlap = false;
    T *aux[2];
    aux[0] = (T *)cm_ensure_aux(m, (size_t)chunk * frame_elems * sizeof(T));
    if (!aux[0]) return CM_ERR_NOMEM;
    aux[1] = aux[0];
    if (overlap) {
        aux[1] = (T *)cm_ensure_aux(m, (size_t)chunk * frame_elems * sizeof(T), 2);
        if (!aux[1]) return CM_ERR_NOMEM;
        if (!m->s2) {
            int lo = 0, hi = 0;
            CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            CUDA_TRY(cudaStreamCreateWithPriority(&m->s2, cudaStreamNonBlocking, hi));
            for (int i = 0; i < 2; ++i) {
                CUDA_TRY(cudaEventCreateWithFlags(&m->ev_p1[i], cudaEventDisableTiming));
                CUDA_TRY(cudaEventCreateWithFlags(&m->ev_p2[i], cudaEventDisableTiming));
            }
        }
    }
    const size_t in_frame = (size_t)io.nrows * p.Wc, out_frame = (size_t)io.nrows * p.Wo * 3;
    int nchunks = 0;
    for (int f0 = 0; f0 < io.nframes; f0 += chunk, ++nchunks) {
        const int buf = nchunks & 1;
        IoArgs<T> c = io;
        c.nframes = io.nframes - f0 < chunk ? io.nframes - f0 : chunk;
        c.first_frame = io.first_frame + f0;
        c.aux = aux[buf];
        if (c.in_u8) c.in_u8 += (size_t)f0 * in_frame;
        if (c.in_f) c.in_f += (size_t)f0 * in_frame;
        if (c.out_u8) c.out_u8 += (size_t)f0 * out_frame;
        if (c.out_f) c.out_f += (size_t)f0 * out_frame;
        if (c.yuv) c.yuv += (size_t)f0 * io.nrows * 3 * p.Wo;
        IoArgs<T> a = c;                      // pass 1 also covers the neighbour rows the combination reads
        a.out_begin = c.out_begin >= 2 ? c.out_begin - 2 : 0;
        int end = c.out_begin + c.out_count + (MODE >= PAIR_NTSC3 ? 2 : 0);
        if (end > c.nrows) end = c.nrows;
        a.out_count = end - a.out_begin;
        if (overlap && nchunks >= 2) CUDA_TRY(cudaStreamWaitEvent(st, m->ev_p2[buf], 0));     // buffer free again
        {
            LaunchTimer lt(m, MODE == PAIR_PALD ? CM_K_PALD : CM_K_COMB, st);
            const int rpc = cm_rows_per_cta(m, (long long)a.out_count * c.nframes);     // rows per CTA: the next row is prefetched while one is filtered (1: 7.97, 2: 7.67, 4: 8.15 us/frame)
            pass1<<<dim3((unsigned)((a.out_count + rpc - 1) / rpc), 1u, (unsigned)c.nframes), threads1, b1, st>>>(p, a);
        }
        cm_count_launch();
        CUDA_TRY(cudaGetLastError());
        cudaStream_t st2 = st;
        if (overlap) {
            CUDA_TRY(cudaEventRecord(m->ev_p1[buf], st));
            CUDA_TRY(cudaStreamWaitEvent(m->s2, m->ev_p1[buf], 0));
            st2 = m->s2;
        }
        {
            LaunchTimer lt(m, CM_K_DECODE_OTHER, st2);
            const int segs = (((c.out_count + 1) >> 1) + CM_SEG - 1) / CM_SEG, threads = 128;
            dim3 grid((unsigned)((segs * (p.W >> 2) + threads - 1) / threads), 2u, (unsigned)c.nframes);
            if (!c.yuv) k_qam_combine<T, MODE, 0><<<grid, threads, 0, st2>>>(p, c);
            else if (MODE >= PAIR_NTSC3 && (p.flags & CM_FLAG_MINAVG)) k_qam_combine<T, MODE, 2><<<grid, threads, 0, st2>>>(p, c);
            else k_qam_combine<T, MODE, 1><<<grid, threads, 0, st2>>>(p, c);
        }
        cm_count_launch();
        CUDA_TRY(cudaGetLastError());
        if (overlap) CUDA_TRY(cudaEventRecord(m->ev_p2[buf], m->s2));
    }
    if (overlap) {          // everything this call produced is ordered before whatever the caller queues next on `st`
        CUDA_TRY(cudaStreamWaitEvent(st, m->ev_p2[(nchunks - 1) & 1], 0));
        if (nchunks >= 2) CUDA_TRY(cudaStreamWaitEvent(st, m->ev_p2[nchunks & 1], 0));
    }
    return CM_OK;
}
#endif

#if CM_PART(1)
template <typename T>
int launch_pald(cm_modem *m, IoArgs<T> io, cudaStream_t st) {
    const DevParams<T> &p = params_of<T>(m);
    if (io.out_count <= 0) return CM_OK;
    if (!io.prof && !m->tune.onepass &&
        (128 + (size_t)p.n1p + 6 * (size_t)p.hb2) * sizeof(T) <= (size_t)m->smem_optin)
        return launch_rows_pair<T, PAIR_PALD>(m, io, st);
    auto bytes = [&](int r) {
        return (CM_TAPS_ELEMS + (size_t)(r + 1) * (p.n1p + 2 * (size_t)p.hb2) + (size_t)r * 4 * p.hb2) * sizeof(T);
    };
    int R = pick_rows(m, 4, (size_t)m->smem_optin / 2, bytes);
    if (!R) R = pick_rows(m, 2, (size_t)m->smem_optin, bytes);
    if (!R) return cm_fail(CM_ERR_UNSUPPORTED, "line too wide for the PAL-D kernel%s");
    const bool teams = needs_teams(p);
    set_groups(io, R);
    int rc = teams ? set_smem(k_pald_combed<T, true>, bytes(R)) : set_smem(k_pald_combed<T, false>, bytes(R));
    if (rc) return rc;
    dim3 grid = cm_grid(io);
    {
        LaunchTimer lt(m, CM_K_PALD, st);
        if (teams) k_pald_combed<T, true><<<grid, CM_NTHREADS, bytes(R), st>>>(p, io);
        else k_pald_combed<T, false><<<grid, cta_threads(m, 2 * R), bytes(R), st>>>(p, io);
    }
    cm_count_launch();
    CUDA_TRY(cudaGetLastError());
    return CM_OK;
}

CM_INSTANTIATE(template int launch_pald<float>(cm_modem *, IoArgs<float>, cudaStream_t);,
               template int launch_pald<double>(cm_modem *, IoArgs<double>, cudaStream_t);)
#endif

#if CM_PART(2)
template <typename T, int MODE>
int launch_comb(cm_modem *m, IoArgs<T> io, cudaStream_t st) {
    const DevParams<T> &p = params_of<T>(m);
    if (io.out_count <= 0) return CM_OK;
    // (the legacy kernels below do not implement avg=minavg)
    if ((!m->tune.onepass || (p.flags & CM_FLAG_MINAVG)) &&
        (128 + (size_t)p.n1p + 6 * (size_t)p.hb2) * sizeof(T) <= (size_t)m->smem_optin)
        return launch_rows_pair<T, MODE == COMB_NTSC2 ? PAIR_NTSC2 : (MODE == COMB_NTSC3 ? PAIR_NTSC3 : PAIR_PAL3)>(m, io, st);
    auto bytes = [&](int r) {
        return (CM_TAPS_ELEMS + (size_t)(r + 2) * (p.n1p + 2 * (size_t)p.hb2) + (size_t)r * 4 * p.hb2) * sizeof(T);
    };
    int R = pick_rows(m, 4, (size_t)m->smem_optin / 2, bytes);
    if (!R) R = pick_rows(m, 2, (size_t)m->smem_optin, bytes);
    if (!R) return cm_fail(CM_ERR_UNSUPPORTED, "line too wide for the comb kernel%s");
    const bool teams = needs_teams(p);
    set_groups(io, R);
    int rc = teams ? set_smem(k_qam_comb<T, MODE, true>, bytes(R)) : set_smem(k_qam_comb<T, MODE, false>, bytes(R));
    if (rc) return rc;
    dim3 grid = cm_grid(io);
    {
        LaunchTimer lt(m, CM_K_COMB, st);
        if (teams) k_qam_comb<T, MODE, true><<<grid, CM_NTHREADS, bytes(R), st>>>(p, io);
        else k_qam_comb<T, MODE, false><<<grid, cta_threads(m, 2 * R), bytes(R), st>>>(p, io);
    }
    cm_count_launch();
    CUDA_TRY(cudaGetLastError());
    return CM_OK;
}

#define CM_COMB_INST(T)                                                                        \
    template int launch_comb<T, COMB_NTSC2>(cm_modem *, IoArgs<T>, cudaStream_t);              \
    template int launch_comb<T, COMB_NTSC3>(cm_modem *, IoArgs<T>, cudaStream_t);              \
    template int launch_comb<T, COMB_PAL3>(cm_modem *, IoArgs<T>, cudaStream_t);
CM_INSTANTIATE(CM_COMB_INST(float), CM_COMB_INST(double))
#endif

#if CM_PART(3)
// Comb decoders with non-default knobs (luma notch, avg=minavg): run the decoder with the (y, u, v) of the rows
// concerned diverted to a scratch, then k_finish_rows.  2-line decoders notch the rows that have a predecessor
// (comb.py:48-55), the 3-line decoders every row they keep (comb.py:96-109, pal.py:191-228); minavg applies to the
// combed rows of the 3-line decoders (the field tops of Pal3DModem keep their band-split chroma).
template <typename T>
static int qam_decode_post(cm_modem *m, IoArgs<T> io, cudaStream_t st) {
    const DevParams<T> &p = params_of<T>(m);
    if (io.out_count <= 0) return CM_OK;
    const bool notch = (p.flags & CM_FLAG_NOTCH) != 0;
    const bool pal3 = p.kind == CM_KIND_PAL_3D && (p.flags & (CM_FLAG_PAL3D_SIN | CM_FLAG_PAL3D_COS));
    const bool three_line = p.kind == CM_KIND_NTSC_3D || pal3;
    const bool minavg = three_line && (p.flags & CM_FLAG_MINAVG) && !(p.flags & CM_FLAG_NTSC_NO_COMB);
    const size_t smem1 = (size_t)p.n1p * sizeof(T), smem3 = 3 * smem1;
    int rc = set_smem(k_finish_rows<T, false>, smem1);
    if (rc) return rc;
    rc = set_smem(k_finish_rows<T, true>, smem3);
    if (rc) return rc;
    const int chunk = io.nframes < 64 ? io.nframes : 64;
    const size_t frame_elems = (size_t)io.nrows * 3 * p.Wo;
    T *yuv = (T *)cm_ensure_aux(m, (size_t)chunk * frame_elems * sizeof(T), 1);
    if (!yuv) return CM_ERR_NOMEM;
    const size_t in_frame = (size_t)io.nrows * p.Wc, out_frame = (size_t)io.nrows * p.Wo * 3;
    auto rows_from = [](IoArgs<T> a, int begin) {            // the rows of a at or below `begin`
        if (a.out_begin < begin) {
            a.out_count -= begin - a.out_begin;
            a.out_begin = begin;
        }
        return a;
    };
    auto rows_before = [](IoArgs<T> a, int end) {
        if (a.out_begin + a.out_count > end) a.out_count = end - a.out_begin;
        return a;
    };
    auto finish = [&](const IoArgs<T> &n, bool remod) -> int {
        if (n.out_count <= 0) return CM_OK;
        const dim3 grid((unsigned)n.out_count, 1u, (unsigned)n.nframes);
        {
            LaunchTimer lt(m, CM_K_DECODE_OTHER, st);
            if (remod) k_finish_rows<T, true><<<grid, CM_ROW_THREADS, smem3, st>>>(p, n);
            else k_finish_rows<T, false><<<grid, CM_ROW_THREADS, smem1, st>>>(p, n);
        }
        cm_count_launch();
        CUDA_TRY(cudaGetLastError());
        return CM_OK;
    };
    for (int f0 = 0; f0 < io.nframes; f0 += chunk) {
        IoArgs<T> c = io;
        c.nframes = io.nframes - f0 < chunk ? io.nframes - f0 : chunk;
        c.first_frame = io.first_frame + f0;
        c.yuv = yuv;
        if (c.in_u8) c.in_u8 += (size_t)f0 * in_frame;
        if (c.in_f) c.in_f += (size_t)f0 * in_frame;
        if (c.out_u8) c.out_u8 += (size_t)f0 * out_frame;
        if (c.out_f) c.out_f += (size_t)f0 * out_frame;
        rc = qam_decode<T>(m, c, CM_MODE_DEFAULT, st);
        if (rc) return rc;
        if (!three_line) {
            rc = finish(rows_from(c, 2), false);                          // notch on the rows with a predecessor
        } else if (!minavg) {
            rc = finish(c, false);                                        // notch on every row
        } else if (pal3) {
            rc = finish(rows_from(c, 2), true);                           // combed rows: re-modulate (+ notch)
            if (!rc && notch) rc = finish(rows_before(c, 2), false);      // field tops: notch only
        } else {
            rc = finish(c, true);
        }
        if (rc) return rc;
    }
    return CM_OK;
}

template <typename T>
int qam_decode(cm_modem *m, IoArgs<T> io, int mode, cudaStream_t st) {
    const DevParams<T> &p = params_of<T>(m);
    if (mode == CM_MODE_BANDSPLIT_NOSTRIP) return launch_bandsplit<T>(m, io, 2, st);
    if (mode == CM_MODE_EXTRACT_CHROMA) return launch_extract<T>(m, io, st);
    const bool pal3 = p.kind == CM_KIND_PAL_3D && (p.flags & (CM_FLAG_PAL3D_SIN | CM_FLAG_PAL3D_COS));
    const bool three_line = p.kind == CM_KIND_NTSC_3D || pal3;
    const bool post = (p.flags & CM_FLAG_NOTCH) || (three_line && (p.flags & CM_FLAG_MINAVG) && !(p.flags & CM_FLAG_NTSC_NO_COMB));
    if (post && p.kind != CM_KIND_QAM_BANDSPLIT && !io.yuv) return qam_decode_post<T>(m, io, st);
    IoArgs<T> top, rest;
    split_top(io, top, rest);
    // field tops: the 2-line decoders bypass the notch there (comb.py:48-49); Pal3DModem's take it but never minavg
    if (!(pal3 && (p.flags & CM_FLAG_NOTCH))) top.yuv = nullptr;
    int rc;
    switch (p.kind) {
        case CM_KIND_QAM_BANDSPLIT:
            return launch_bandsplit<T>(m, io, 0, st);
        case CM_KIND_PAL_D:
            rc = launch_bandsplit<T>(m, top, 0, st);
            return rc ? rc : launch_pald<T>(m, rest, st);
        case CM_KIND_NTSC_COMB:
            rc = launch_bandsplit<T>(m, top, 0, st);
            if (rc) return rc;
            if (p.flags & CM_FLAG_NTSC_NO_COMB)      // ntsc.py:71-72: chroma of the row itself, luma = c - remod
                return launch_bandsplit<T>(m, rest, 1, st);
            return launch_comb<T, COMB_NTSC2>(m, rest, st);
        case CM_KIND_NTSC_3D:
            if (p.flags & CM_FLAG_NTSC_NO_COMB) return launch_bandsplit<T>(m, io, 1, st);
            return launch_comb<T, COMB_NTSC3>(m, io, st);
        case CM_KIND_PAL_3D:
            if (!(p.flags & (CM_FLAG_PAL3D_SIN | CM_FLAG_PAL3D_COS))) {   // pal.py:181-182: plain PAL-D
                rc = launch_bandsplit<T>(m, top, 0, st);
                return rc ? rc : launch_pald<T>(m, rest, st);
            }
            rc = launch_bandsplit<T>(m, top, 1, st);
            return rc ? rc : launch_comb<T, COMB_PAL3>(m, rest, st);
        default:
            return cm_fail(CM_ERR_UNSUPPORTED, "decode: not a QAM kind%s");
    }
}

CM_INSTANTIATE(template int qam_decode<float>(cm_modem *, IoArgs<float>, int, cudaStream_t);,
               template int qam_decode<double>(cm_modem *, IoArgs<double>, int, cudaStream_t);)
#endif
