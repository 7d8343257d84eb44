// Launchers of the 3x-oversampled AM families: NIIR / SECAM-IV (cm_niir.cuh) and 819-line proto-SECAM (cm_proto.cuh).
#include "cm_host.h"
#include "cm_niir.cuh"
#include "cm_proto.cuh"

template <typename T, class K, class F>
static int launch_rows(cm_modem *m, IoArgs<T> io, cudaStream_t st, K kernel, F bytes, int rmax, int warps_per_row,
                       int extra_rows, int timer_id, const char *what) {
    if (io.out_count <= 0) return CM_OK;
    int R = pick_rows(m, rmax, (size_t)m->smem_optin / 2, bytes);
    if (!R) R = pick_rows(m, 1, (size_t)m->smem_optin, bytes);
    if (!R) return cm_fail(CM_ERR_UNSUPPORTED, "line too wide for the %s kernel", what);
    set_groups(io, R);
    int rc = set_smem(kernel, bytes(R));
    if (rc) return rc;
    dim3 grid = cm_grid(io);
    int threads = cta_threads(m, warps_per_row * (R + extra_rows));
    // cm_tune::min_warps may ask for more warps than the kernel is compiled for (k_niir_decode: 192 threads); the teams
    // take whatever warps the CTA has, and a launch above the bound fails
    cudaFuncAttributes fa;
    CUDA_TRY(cudaFuncGetAttributes(&fa, kernel));
    if (threads > fa.maxThreadsPerBlock) threads = fa.maxThreadsPerBlock & ~31;
    {
        LaunchTimer lt(m, timer_id, st);
        kernel<<<grid, threads, bytes(R), st>>>(params_of<T>(m), io);
    }
    cm_count_launch();
    CUDA_TRY(cudaGetLastError());
    return CM_OK;
}

template <typename T>
int niir_encode(cm_modem *m, IoArgs<T> io, cudaStream_t st) {
    const DevParams<T> &p = params_of<T>(m);
    if (io.in_u8 && p.enc_geo && !m->tune.rows_v1 && !m->tune.onepass) {           // strips of rows, one at a time (k_niir_encode2)
        if (io.out_count <= 0) return CM_OK;
        void (*kern)(const DevParams<T>, const IoArgs<T>) =
            p.enc_geo == 1 ? k_niir_encode2<T, 1> : (p.enc_geo == 2 ? k_niir_encode2<T, 2> : k_niir_encode2<T, 3>);
        const size_t b2 = (128 + 7 * (size_t)p.n1p) * sizeof(T);
        int rc = set_smem(kern, b2);
        if (rc) return rc;
        // rows per strip: the averaging / hue-correcting front ends fetch one row more than the strip is long, so long strips
        // are cheaper — as long as the grid still fills the chip (8 CTAs of 2 warps per SM, two waves)
        const long long rows_total = (long long)io.out_count * io.nframes;
        int R = (int)(rows_total / (16LL * m->sm_count));
        R = R < 1 ? 1 : (R > 16 ? 16 : R);
        if (m->tune.rows_max > 0) R = m->tune.rows_max;
        set_groups(io, R);
        const int nf = (io.out_count + 1) >> 1;
        {
            LaunchTimer lt(m, CM_K_ENCODE, st);
            kern<<<dim3((unsigned)((nf + R - 1) / R), 2u, (unsigned)io.nframes), p.enc_geo == 1 ? 64 : 128, b2, st>>>(p, io);
        }
        cm_count_launch();
        CUDA_TRY(cudaGetLastError());
        return CM_OK;
    }
    auto bytes = [&](int r) { return (size_t)r * 3 * p.n1p * sizeof(T); };
    return launch_rows<T>(m, io, st, k_niir_encode<T>, bytes, 1, 2, 0, CM_K_ENCODE, "NIIR encode");
}

template <typename T>
int niir_decode(cm_modem *m, IoArgs<T> io, cudaStream_t st) {
    const DevParams<T> &p = params_of<T>(m);
    if (p.row_geo && !m->tune.rows_v1 && !m->tune.onepass) {           // strips of rows, one at a time (k_niir_decode2)
        if (io.out_count <= 0) return CM_OK;
        const size_t b2 = (128 + 2 * (size_t)p.n1p + 9 * (size_t)p.hb3) * sizeof(T);
        if (b2 <= (size_t)m->smem_optin) {
            void (*kern)(const DevParams<T>, const IoArgs<T>) = p.row_geo == 1 ? k_niir_decode2<T, 1> : k_niir_decode2<T, 3>;
            int rc = set_smem(kern, b2);
            if (rc) return rc;
            // rows per strip: the row before a strip is recomputed, so long strips are cheaper — as long as the grid
            // still fills the chip (6 CTAs per SM)
            const long long rows_total = (long long)io.out_count * io.nframes;
            int R = (int)(rows_total / (6LL * m->sm_count));
            R = R < 2 ? 2 : (R > 12 ? 12 : R);
            if (m->tune.rows_max > 0) R = m->tune.rows_max;
            set_groups(io, R);
            {
                LaunchTimer lt(m, CM_K_DECODE_OTHER, st);
                kern<<<cm_grid(io), p.row_geo == 1 ? 64 : 128, b2, st>>>(p, io);
            }
            cm_count_launch();
            CUDA_TRY(cudaGetLastError());
            return CM_OK;
        }
    }
    auto bytes = [&](int r) { return (128 + (size_t)(r + 1) * (p.n1p + 9 * (size_t)p.hb3)) * sizeof(T); };
    return launch_rows<T>(m, io, st, k_niir_decode<T>, bytes, 2, 2, 1, CM_K_DECODE_OTHER, "NIIR decode");
}

template <typename T>
int proto_encode(cm_modem *m, IoArgs<T> io, cudaStream_t st) {
    const DevParams<T> &p = params_of<T>(m);
    if (io.in_u8 && p.row_geo && !m->tune.rows_v1 && !m->tune.onepass) {
        if (io.out_count <= 0) return CM_OK;
        void (*kern)(const DevParams<T>, const IoArgs<T>) = p.row_geo == 1 ? k_proto_encode_row2<T, 1> : k_proto_encode_row2<T, 3>;
        const size_t b2 = (128 + 2 * (size_t)p.n1p + 3 * (size_t)p.hb3) * sizeof(T);
        if (b2 <= (size_t)m->smem_optin) {
            int rc = set_smem(kern, b2);
            if (rc) return rc;
            const int rpc = cm_rows_per_cta(m, (long long)io.out_count * io.nframes), nf = (io.out_count + 1) >> 1;
            {
                LaunchTimer lt(m, CM_K_ENCODE, st);
                kern<<<dim3((unsigned)((nf + rpc - 1) / rpc), 2u, (unsigned)io.nframes), p.row_geo == 1 ? 128 : 256, b2, st>>>(p, io);
            }
            cm_count_launch();
            CUDA_TRY(cudaGetLastError());
            return CM_OK;
        }
    }
    auto bytes = [&](int r) { return (128 + (size_t)r * (2 * (size_t)p.n1p + 3 * (size_t)p.hb3)) * sizeof(T); };
    return launch_rows<T>(m, io, st, k_proto_encode<T>, bytes, 1, 2, 0, CM_K_ENCODE, "proto-SECAM encode");
}

template <typename T>
int proto_decode(cm_modem *m, IoArgs<T> io, cudaStream_t st) {
    const DevParams<T> &p = params_of<T>(m);
    if (io.out_count <= 0) return CM_OK;
    // pass 1 (heavy): (luma, X) per row for the output rows and the two rows above them, into a pairing scratch of
    // 2 * Wo elements per row; the batch is cut so that the scratch stays within 2 GiB
    const size_t frame_elems = (size_t)io.nrows * 2 * p.Wo;
    int chunk = (int)(((size_t)2 << 30) / (frame_elems * sizeof(T)));
    if (chunk < 1) chunk = 1;
    if (m->tune.chunk > 0) chunk = m->tune.chunk;
    if (chunk > io.nframes) chunk = io.nframes;
    T *aux = (T *)cm_ensure_aux(m, (size_t)chunk * frame_elems * sizeof(T));
    if (!aux) return CM_ERR_NOMEM;
    const size_t b2 = (128 + (size_t)p.n1p + 6 * (size_t)p.hb3) * sizeof(T);
    const bool rows2 = p.row_geo && !m->tune.rows_v1 && !m->tune.onepass && b2 <= (size_t)m->smem_optin;
    void (*kern)(const DevParams<T>, const IoArgs<T>) = p.row_geo == 1 ? k_proto_decode2<T, 1> : k_proto_decode2<T, 3>;
    if (rows2) {
        int rc = set_smem(kern, b2);
        if (rc) return rc;
    }
    auto bytes = [&](int r) { return (128 + (size_t)r * (p.n1p + 9 * (size_t)p.hb3)) * sizeof(T); };
    const size_t in_frame = (size_t)io.nrows * p.Wc, out_frame = (size_t)io.nrows * p.Wo * 3;
    for (int f0 = 0; f0 < io.nframes; f0 += chunk) {
        IoArgs<T> c = io;
        c.nframes = io.nframes - f0 < chunk ? io.nframes - f0 : chunk;
        c.first_frame = io.first_frame + f0;
        c.aux = aux;
        if (c.in_u8) c.in_u8 += (size_t)f0 * in_frame;
        if (c.in_f) c.in_f += (size_t)f0 * in_frame;
        if (c.out_u8) c.out_u8 += (size_t)f0 * out_frame;
        if (c.out_f) c.out_f += (size_t)f0 * out_frame;
        IoArgs<T> a = c;
        a.out_begin = c.out_begin >= 2 ? c.out_begin - 2 : 0;
        a.out_count = c.out_begin + c.out_count - a.out_begin;
        if (rows2) {
            const int rpc = cm_rows_per_cta(m, (long long)a.out_count * c.nframes);
            {
                LaunchTimer lt(m, CM_K_DECODE_OTHER, st);
                kern<<<dim3((unsigned)((a.out_count + rpc - 1) / rpc), 1u, (unsigned)c.nframes), p.row_geo == 1 ? 128 : 256, b2, st>>>(p, a);
            }
            cm_count_launch();
            CUDA_TRY(cudaGetLastError());
        } else {
            // two tasks per row (chroma, luma), each run by a team of up to four warps
            int rc = launch_rows<T>(m, a, st, k_proto_decode<T>, bytes, 2, 4, 0, CM_K_DECODE_OTHER, "proto-SECAM decode");
            if (rc) return rc;
        }
        // pass 2 (light): pair rows y / y-2, inverse matrix, store
        {
            LaunchTimer lt(m, CM_K_DECODE_OTHER, st);
            dim3 grid(1u, (unsigned)c.out_count, (unsigned)c.nframes);
            k_pair_rows_store<T><<<grid, 192, 0, st>>>(p, c);
        }
        cm_count_launch();
        CUDA_TRY(cudaGetLastError());
    }
    return CM_OK;
}

#define CM_INST(fn)                                                                     \
    CM_INSTANTIATE(template int fn<float>(cm_modem *, IoArgs<float>, cudaStream_t);,     \
                   template int fn<double>(cm_modem *, IoArgs<double>, cudaStream_t);)
CM_INST(niir_encode)
CM_INST(niir_decode)
CM_INST(proto_encode)
CM_INST(proto_decode)
