// PAL-D decode as a banded matrix product on the tensor cores (k_pald_mma): one kernel from the u8 composite to RGB.
//
// For one row, pass 1 of the two-pass decoder (k_qam_rows2<PALD>) is a fixed linear map from the composite row to the
// four planes (a', b', LPpre a', LPpre b') before the row's own phase rotation: the carrier comes from a row-independent
// table, the rotation is applied afterwards, and the level map u8 -> signal is affine.  The host builds that map in
// float64 from the handle's filters (cm_api.cu: plan_pald_mma) and keeps its band: output sample x depends on the inputs
// [x - KPRE, x + KW - KPRE - TS] only (to 2^-26 of the largest coefficient).  For a tile of TS output samples the map is
// a [KW x 4 TS] block B, split into two FP16 terms hi + lo with a power-of-two scale per column; the composite bytes
// are exact in FP16.  So for 128 rows at once
//     planes[128 x 4 TS] = (X[128 x KW] . (B_hi + B_lo)) * scale^-1 + bias
// is two K-loops of tcgen05.mma kind::f16 with FP32 accumulation in tensor memory (lane = row).  The epilogue does
// what k_qam_combine<PALD> does with the planes of a row and of its predecessor in the field: rotation to the row's
// phase, pair_uv, re-modulation, the colour matrix and the store.
//
// Rows.  The rows of a call are listed field by field and frame by frame; each field starts with the predecessor of
// its first output row (computed, never stored).  Tile rb holds list entries 127 rb - 1 .. 127 rb + 126: lane 0 is a
// halo row whose planes only serve lane 1 as its predecessor.  A CTA keeps one column tile (its B in shared memory,
// loaded once by one bulk copy) and walks row tiles; the MMA of the next row tile runs under the epilogue of the
// current one (two accumulators in tensor memory, two A buffers).
//
// Compiled for float only (the float64 build keeps the two-pass kernels).
#include <cuda_fp16.h>

#include "cm_host.h"
#include "cm_qam.cuh"

#if !defined(CM_INST_F64)

namespace {

constexpr int kThreads = 512;                 // 16 warps: warp w reads TMEM lanes 32 (w % 4) .., samples 8 (w / 4) ..
constexpr int kRows = 128;                    // UMMA M: rows per tile, TMEM lane = row
constexpr int kOut = kRows - 1;               // rows a tile outputs (lane 0 is the halo)
constexpr int kABytes = CM_PALD_KW * kRows * 2;            // one A buffer: [KW / 8][128 rows][8 halves]
constexpr int kBTerm = CM_PALD_KW * CM_PALD_N * 2;         // one term of B: [KW / 8][N][8 halves]
constexpr int kSmemB = 0, kSmemA = 2 * kBTerm, kSmemX = kSmemA + 2 * kABytes;
constexpr int kSmemCS = kSmemX + 16 * 32 * 4 * 8;         // lane 31 of each warp: 8 samples x 4 planes
constexpr int kSmemBar = kSmemCS + 2 * CM_PALD_N * 4;
constexpr int kSmemBytes = kSmemBar + 64;
constexpr int kTmemCols = 2 * CM_PALD_N;
static_assert(CM_PALD_TS == 32 && CM_PALD_N == 128, "the epilogue maps 16 warps onto 4 x 32 lanes and 4 x 8 samples");
static_assert(kSmemBytes <= 227 * 1024, "shared memory");

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// UMMA shared-memory descriptor, no swizzle, K-major: core matrices of 8 rows x 16 bytes; LBO = byte distance of
// neighbouring core matrices along K, SBO = along M / N; bits 46-48 = 0b001 (tcgen05 descriptor version)
__device__ __forceinline__ uint64_t umma_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((addr >> 4) & 0x3fff) | ((uint64_t)((lbo >> 4) & 0x3fff) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3fff) << 32) | (1ull << 46);
}
// instruction descriptor of kind::f16: D F32, A / B F16, both K-major, N >> 3 at bit 17, M >> 4 at bit 24
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(CM_PALD_N >> 3) << 17) | ((uint32_t)(kRows >> 4) << 24);

__device__ __forceinline__ void mbar_init(uint32_t bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, unsigned parity) {
    uint32_t done = 0;
    while (!done)
        asm volatile(
            "{\n\t.reg .pred P;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, P;\n}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
}

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t a, uint64_t b, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d),
        "l"(a), "l"(b), "r"(kIdesc), "r"(accumulate));
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 32 consecutive TMEM columns of this thread's lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float v[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,"
        "%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// u8 quad -> four FP16 (exact): 0x64XX is 1024 + XX
__device__ __forceinline__ uint2 u8x4_to_h4(uint32_t w) {
    const __half2 k1024 = __half2half2(__ushort_as_half((unsigned short)0x6400));
    const uint32_t pl = __byte_perm(w, 0x64646464u, 0x4140), ph = __byte_perm(w, 0x64646464u, 0x4342);
    __half2 lo = __hsub2(*reinterpret_cast<const __half2 *>(&pl), k1024);
    __half2 hi = __hsub2(*reinterpret_cast<const __half2 *>(&ph), k1024);
    return make_uint2(*reinterpret_cast<uint32_t *>(&lo), *reinterpret_cast<uint32_t *>(&hi));
}

struct RowRef {
    long long off;      // byte offset of the row in the composite batch; < 0: no row (padding of the last tile)
    int f, row;         // frame of the batch, buffer row
    bool out;           // an output row (not the predecessor that opens a field)
};

__device__ __forceinline__ RowRef list_row(const PaldMmaArgs &g, const IoArgs<float> &io, long long i, int Wc) {
    RowRef r{-1, 0, 0, false};
    if (i < 0 || i >= g.total) return r;
    const int f = (int)(i / g.per_frame);
    int j = (int)(i - (long long)f * g.per_frame);
    int k = j, row0 = g.row_a;
    if (j >= g.len_a) { k = j - g.len_a; row0 = g.row_a + 1; }
    r.f = f;
    r.row = row0 + 2 * k;
    r.out = k > 0;
    r.off = ((long long)f * io.nrows + r.row) * Wc;
    return r;
}

}  // namespace

__global__ void __launch_bounds__(kThreads, 1)
k_pald_mma(const __grid_constant__ DevParams<float> p, const __grid_constant__ IoArgs<float> io,
           const __grid_constant__ PaldMmaArgs g) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int W = p.W, Wc = p.Wc;
    const int tile = blockIdx.y, x0 = tile * CM_PALD_TS;
    float *xbuf = reinterpret_cast<float *>(smem + kSmemX);
    float *cs = reinterpret_cast<float *>(smem + kSmemCS);              // [inverse scale | bias] per column
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kSmemBar);     // [0] B loaded, [1], [2] MMA done per buffer
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + kSmemBar + 32);
    const uint32_t bar_b = smem_u32(bars), bar_mma0 = smem_u32(bars + 1);

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 0) {
        mbar_init(bar_b, 1);
        mbar_init(bar_mma0, 1);
        mbar_init(bar_mma0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // B of this column tile: both terms, already in the canonical layout
        const unsigned char *src = reinterpret_cast<const unsigned char *>(g.b) + (size_t)tile * 2 * kBTerm;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_b), "r"(2 * kBTerm) : "memory");
        constexpr int kPiece = 16384;
        for (int o = 0; o < 2 * kBTerm; o += kPiece)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             smem_u32(smem + kSmemB + o)),
                         "l"(src + o), "r"(kPiece), "r"(bar_b)
                         : "memory");
    }
    for (int i = tid; i < 2 * CM_PALD_N; i += kThreads) cs[i] = g.cs[(size_t)tile * 2 * CM_PALD_N + i];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    // staging: thread tid stages row (tid & 127) of the tile, K-chunks (tid >> 7) + 4 it, it = 0 .. 4 (8 samples each)
    constexpr int kChunks = CM_PALD_KW / 8, kIt = kChunks / 4;
    static_assert(kChunks % 4 == 0, "K chunks per staging thread");
    const int srow = tid & (kRows - 1), schunk = tid >> 7;
    uint32_t pw[2 * kIt];
    auto fetch = [&](int rb) {
        const RowRef r = list_row(g, io, (long long)rb * kOut + srow - 1, Wc);
#pragma unroll
        for (int it = 0; it < kIt; ++it)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int x = x0 - CM_PALD_KPRE + 8 * (schunk + 4 * it) + 4 * h;
                pw[2 * it + h] = (r.off >= 0 && x >= 0 && x < W)
                                     ? __ldg(reinterpret_cast<const uint32_t *>(io.in_u8 + r.off + x))
                                     : 0u;
            }
    };
    auto stage = [&](int buf) {
        unsigned char *a = smem + kSmemA + buf * kABytes;
#pragma unroll
        for (int it = 0; it < kIt; ++it) {
            const uint2 l = u8x4_to_h4(pw[2 * it]), h = u8x4_to_h4(pw[2 * it + 1]);
            *reinterpret_cast<uint4 *>(a + (schunk + 4 * it) * (kRows * 16) + srow * 16) = make_uint4(l.x, l.y, h.x, h.y);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    };
    auto issue = [&](int buf) {      // one thread: hi then lo term into accumulator `buf`
        const uint32_t a = smem_u32(smem + kSmemA + buf * kABytes), b = smem_u32(smem + kSmemB);
        const uint32_t d = tmem + (uint32_t)(buf * CM_PALD_N);
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
            for (int ks = 0; ks < CM_PALD_KW / 16; ++ks)
                umma_f16(d, umma_desc(a + ks * 2 * (kRows * 16), kRows * 16, 128),
                         umma_desc(b + t * kBTerm + ks * 2 * (CM_PALD_N * 16), CM_PALD_N * 16, 128), (t | ks) != 0);
        umma_commit(bar_mma0 + 8 * buf);
    };

    // epilogue constants
    PairCoef<float> kc;
    Real<float>::sincos_turns(p.line_shift, kc.sl, kc.cl);
    kc.sf = p.scalars[QS_PALD_SIN];
    kc.cf = p.scalars[QS_PALD_COS];
    float rs, rc;
    Real<float>::sincos_turns(p.phases[QP_STEP1X], rs, rc);
    const int quarter = warp & 3, sg = warp >> 2;         // TMEM lanes 32 quarter .., samples x0 + 8 sg ..
    const int erow = 32 * quarter + lane;

    int rb = blockIdx.x;
    if (rb < g.nblocks) {
        fetch(rb);
        stage(0);
        if (rb + (int)gridDim.x < g.nblocks) fetch(rb + gridDim.x);
    }
    __syncthreads();
    if (tid == 0) {
        mbar_wait(bar_b, 0);           // also when this CTA has no row tile: no bulk copy outlives the CTA
        tc_fence_after();
        if (rb < g.nblocks) issue(0);
    }
    for (int it = 0; rb < g.nblocks; ++it, rb += gridDim.x) {
        const int buf = it & 1;
        const int rbn = rb + gridDim.x;
        if (rbn < g.nblocks) stage(buf ^ 1);       // its previous readers (MMA it-1, epilogue it-1) are done
        tc_fence_before();
        __syncthreads();
        if (rbn < g.nblocks) {
            if (tid == 0) {
                tc_fence_after();
                issue(buf ^ 1);
            }
            if (rbn + (int)gridDim.x < g.nblocks) fetch(rbn + gridDim.x);
        }
        mbar_wait(bar_mma0 + 8 * buf, (it >> 1) & 1);
        tc_fence_after();

        // ---- epilogue of row tile rb: this thread's row, 8 samples ----
        const RowRef r = list_row(g, io, (long long)rb * kOut + erow - 1, Wc);
        const long long frame = io.first_frame + r.f;
        const int line = io.y0 + r.row;
        const unsigned long long sp = start_phase(p, frame, line);
        float v[32];
        tmem_ld32(tmem + ((uint32_t)(32 * quarter) << 16) + (uint32_t)(buf * CM_PALD_N + 32 * sg), v);
        {
            float sphi, cphi;
            Real<float>::sincos_turns(sp + p.phases[QP_BP_SHIFT] - p.phases[QP_HALF_LS], sphi, cphi);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float q[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int n = 32 * sg + 4 * j + c;
                    q[c] = fmaf(v[4 * j + c], cs[n], cs[CM_PALD_N + n]);
                }
                // rotation to the row's own phase (as in k_qam_rows2): (a, b) and (alpha, beta)
                v[4 * j + 0] = fmaf(cphi, q[0], sphi * q[1]);
                v[4 * j + 1] = fmaf(cphi, q[1], -(sphi * q[0]));
                v[4 * j + 2] = fmaf(cphi, q[2], sphi * q[3]);
                v[4 * j + 3] = fmaf(cphi, q[3], -(sphi * q[2]));
            }
        }
        if (lane == 31) {
#pragma unroll
            for (int i = 0; i < 32; ++i) xbuf[warp * 32 + i] = v[i];
        }
        __syncthreads();
        // composite bytes of this row at the tile's samples x0 + 8 sg .. + 8 (FP16 in the A buffer, K offset KPRE + 8 sg)
        const uint4 cw = *reinterpret_cast<const uint4 *>(smem + kSmemA + buf * kABytes +
                                                          ((CM_PALD_KPRE >> 3) + sg) * (kRows * 16) + erow * 16);
        const bool alt = is_alternate(p, frame, line);
        const bool neg = (p.flags & 1) && alt;
        const bool out = r.out && erow > 0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int x = x0 + 8 * sg + 4 * h;
            float y[4], u[4], vv[4], s[4], co[4];
            carrier4(sp + (unsigned long long)x * p.phases[QP_STEP1X], rs, rc, s, co);
            const uint32_t cwh[2] = {h ? cw.z : cw.x, h ? cw.w : cw.y};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int j = 4 * h + i;
                float pv[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float up = __shfl_up_sync(0xffffffffu, v[4 * j + c], 1);
                    pv[c] = lane ? up : (quarter ? xbuf[(warp - 1) * 32 + 4 * j + c] : 0.f);
                }
                const __half2 hc = *reinterpret_cast<const __half2 *>(&cwh[i >> 1]);
                const float byte = (i & 1) ? __high2float(hc) : __low2float(hc);
                const float cc = (5.0f * Real<float>::from_u8((unsigned)byte) - 1.0f) * (float)(1.0 / 3.0);
                float ul, vl;
                pair_uv<float, PAIR_PALD, false>(kc, true, true, alt, pv[0], pv[1], v[4 * j], v[4 * j + 1], 0.f, 0.f, u[i],
                                                 vv[i]);
                pair_uv<float, PAIR_PALD, false>(kc, true, true, alt, pv[2], pv[3], v[4 * j + 2], v[4 * j + 3], 0.f, 0.f, ul,
                                                 vl);
                y[i] = cc - (s[i] * ul + co[i] * (neg ? -vl : vl));
            }
            if (out && x < W) store_rgb4_direct(p, io, r.f, r.row, x, y, u, vv);
        }
        tc_fence_before();
        __syncthreads();            // A buffer `buf`, accumulator `buf` and xbuf are free again
    }
    tc_fence_after();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols));
}

// Rows [out_begin, out_begin + out_count) of every frame (out_begin >= 2: every row has its predecessor in the buffer).
int launch_pald_mma(cm_modem *m, IoArgs<float> io, cudaStream_t st) {
    const DevParams<float> &p = m->pf;
    if (io.out_count <= 0) return CM_OK;
    PaldMmaArgs g;
    g.b = (const uint16_t *)m->d_mma_b;
    g.cs = (const float *)m->d_mma_cs;
    g.row_a = io.out_begin - 2;
    const int na = (io.out_count + 1) >> 1, nb = io.out_count >> 1;
    g.len_a = na + 1;
    g.per_frame = g.len_a + (nb ? nb + 1 : 0);
    g.total = (long long)g.per_frame * io.nframes;
    const long long nblocks = (g.total + kOut - 1) / kOut;
    if (nblocks > 0x7fffffffLL) return cm_fail(CM_ERR_UNSUPPORTED, "batch too large for the PAL-D tensor-core kernel%s");
    g.nblocks = (int)nblocks;
    const int ntiles = (p.W + CM_PALD_TS - 1) / CM_PALD_TS;
    // one CTA per SM (shared memory), a single wave: a column tile per grid row, row tiles strided over grid columns
    long long gx = (long long)m->sm_count / ntiles;
    if (gx > g.nblocks) gx = g.nblocks;
    if (gx < 1) gx = 1;
    int rc = set_smem(k_pald_mma, kSmemBytes);
    if (rc) return rc;
    {
        LaunchTimer lt(m, CM_K_PALD, st);
        k_pald_mma<<<dim3((unsigned)gx, (unsigned)ntiles, 1u), kThreads, kSmemBytes, st>>>(p, io, g);
    }
    cm_count_launch();
    CUDA_TRY(cudaGetLastError());
    return CM_OK;
}

#endif
