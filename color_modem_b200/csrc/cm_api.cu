// C ABI of color_modem_b200 (include/color_modem_b200.h): handle management, filter-table construction and
// dispatch to the per-family launchers (cm_qam.cu, cm_secam.cu, ...).  Host code only.
#include <cuda_fp16.h>
#include <math.h>
#include <stdio.h>

#include <atomic>
#include <new>

#include "cm_host.h"
#include "cm_iir.cuh"
#include "cm_slots.h"

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

int cm_fail(int code, const char *fmt, const char *detail) {
    snprintf(g_err, sizeof(g_err), fmt, detail);
    return code;
}
void cm_count_launch() { g_launches++; }
static int fail(int code, const char *fmt, const char *detail = "") { return cm_fail(code, fmt, detail); }

// ------------------------------------------------------------------------------------------------------------
// filter tables (float64 on the host, cast to the handle's precision)
// ------------------------------------------------------------------------------------------------------------
static void mat_mul(const double a[4], const double b[4], double out[4]) {
    double r[4] = {a[0] * b[0] + a[1] * b[2], a[0] * b[1] + a[1] * b[3], a[2] * b[0] + a[3] * b[2],
                   a[2] * b[1] + a[3] * b[3]};
    memcpy(out, r, sizeof(r));
}

// Chunk length per lane: the kernels instantiate warp_iir for a few compile-time values per rate
// (cm_iir.cuh: warp_iir); pick the one that wastes the least padding, preferring longer chunks on ties.
static void pick_chunk(int rate, int total, int &L, int &nsuper) {
    static const int c1[] = {47, 31, 23}, c2[] = {50, 46, 30}, c3[] = {45, 39, 33};
    const int *cand = rate == 1 ? c1 : (rate == 2 ? c2 : c3);
    const int ncand = 3;
    long best = -1;
    for (int i = 0; i < ncand; ++i) {
        int ns = (total + 32 * cand[i] - 1) / (32 * cand[i]);
        if (ns < 1) ns = 1;
        long padded = (long)ns * 32 * cand[i];
        if (best < 0 || padded < best) { best = padded; L = cand[i]; nsuper = ns; }
    }
}

void cm_build_filter_table(const cm_filter &f, FiltHdr &h, std::vector<double> &tab);
static void build_filter(const cm_filter &f, FiltHdr &h, std::vector<double> &tab) { cm_build_filter_table(f, h, tab); }

static void build_filter_L(const cm_filter &f, FiltHdr &h, std::vector<double> &tab, int L, int nsuper, int lanes);

void cm_build_filter_table(const cm_filter &f, FiltHdr &h, std::vector<double> &tab) {
    int L = 0, nsuper = 0;
    pick_chunk(f.rate, f.n + f.shift, L, nsuper);
    build_filter_L(f, h, tab, L, nsuper, 32);
}

// lanes: chunks per super-chunk (32 for one warp; 32 * team size for the packed team path, where nsuper == 1)
static void build_filter_L(const cm_filter &f, FiltHdr &h, std::vector<double> &tab, int L, int nsuper, int lanes) {
    h.nsec = f.nsec;
    h.shift = f.shift;
    h.n = f.n;
    h.L = L;
    h.nsuper = nsuper;
    h.rate = f.rate;
    h.npad = lanes * L * nsuper;
    h.off = (int)tab.size();
    for (int s = 0; s < f.nsec; ++s) {
        const double *c = f.sos[s];
        std::vector<double> sec(CM_SEC_STRIDE, 0.0);
        for (int i = 0; i < 5; ++i) sec[i] = c[i];
        const double A[4] = {-c[3], -c[4], 1.0, 0.0};     // (y[-1], y[-2]) -> one step of the homogeneous recursion
        double M[4] = {1.0, 0.0, 0.0, 1.0};
        for (int i = 0; i < L; ++i) {                     // M = A^L
            double Q[4];
            mat_mul(A, M, Q);
            memcpy(M, Q, sizeof(M));
        }
        {   // packed fp32 path (two half-chunks per lane): A^ceil(L/2), A^floor(L/2)
            double Mh[4] = {1.0, 0.0, 0.0, 1.0};
            for (int i = 0; i < (L + 1) / 2; ++i) {
                if (i == L / 2) memcpy(&sec[CM_SEC_MHALF + 4], Mh, sizeof(Mh));
                double Q[4];
                mat_mul(A, Mh, Q);
                memcpy(Mh, Q, sizeof(Mh));
            }
            memcpy(&sec[CM_SEC_MHALF], Mh, sizeof(Mh));
            if ((L & 1) == 0) memcpy(&sec[CM_SEC_MHALF + 4], Mh, sizeof(Mh));
        }
        for (int k = 0; k < 5; ++k) {                     // M, M^2, M^4, M^8, M^16
            for (int i = 0; i < 4; ++i) sec[CM_SEC_MPOW + 4 * k + i] = M[i];
            double Q[4];
            mat_mul(M, M, Q);
            memcpy(M, Q, sizeof(M));
        }
        {   // DF-I tables of the packed multi-warp path (team_iir_pk): (A^L)^t per lane, (A^L)^32 per warp
            double Ml[4] = {1.0, 0.0, 0.0, 1.0};
            for (int i = 0; i < L; ++i) {
                double Q[4];
                mat_mul(A, Ml, Q);
                memcpy(Ml, Q, sizeof(Ml));
            }
            double Pw[4] = {1.0, 0.0, 0.0, 1.0};
            for (int t = 0; t < 32; ++t) {
                for (int i = 0; i < 4; ++i) sec[CM_SEC_D_LANE + 4 * t + i] = Pw[i];
                double Q[4];
                mat_mul(Ml, Pw, Q);
                memcpy(Pw, Q, sizeof(Pw));
            }
            for (int i = 0; i < 4; ++i) sec[CM_SEC_D_M32 + i] = Pw[i];
        }
        // DF-II-T tables of the multi-warp path: state (s1, s2), one step = [[-a1, 1], [-a2, 0]]
        const double At[4] = {-c[3], 1.0, -c[4], 0.0};
        double Mt[4] = {1.0, 0.0, 0.0, 1.0};
        for (int i = 0; i < L; ++i) {
            double Q[4];
            mat_mul(At, Mt, Q);
            memcpy(Mt, Q, sizeof(Mt));
        }
        double Pw[4] = {1.0, 0.0, 0.0, 1.0};              // (A^L)^t
        for (int t = 0; t < 32; ++t) {
            for (int i = 0; i < 4; ++i) sec[CM_SEC_T_LANE + 4 * t + i] = Pw[i];
            double Q[4];
            mat_mul(Mt, Pw, Q);
            memcpy(Pw, Q, sizeof(Pw));
        }
        for (int i = 0; i < 4; ++i) sec[CM_SEC_T_M32 + i] = Pw[i];      // (A^L)^32
        double Sq[4];
        memcpy(Sq, Mt, sizeof(Sq));
        for (int k = 0; k < 5; ++k) {
            for (int i = 0; i < 4; ++i) sec[CM_SEC_T_MPOW + 4 * k + i] = Sq[i];
            double Q[4];
            mat_mul(Sq, Sq, Q);
            memcpy(Sq, Q, sizeof(Sq));
        }
        tab.insert(tab.end(), sec.begin(), sec.end());
    }
}

// Geometry of k_qam_rows2 (cm_qam.cuh: RowL<1..3>) for this line length: the first one whose teams cover the three IIR
// use-sites with the chunk lengths compiled for it; fills the QF_ROW_* headers and section tables.  0: none fits.
// Geometry of k_qam_encode_row2 (cm_qam.cuh) for this line length: 1 = 2 warps / 23 samples per lane, 2 = 4 warps / 23,
// 3 = 4 warps / 31; fills the QF_ENC_PRE header.  0: none fits (the multi-row encoder serves the line).
static int plan_encode_kernel(const cm_desc &d, FiltHdr *fh, std::vector<double> &tab) {
    const bool qam = d.kind >= CM_KIND_QAM_BANDSPLIT && d.kind <= CM_KIND_PAL_3D;
    if (!qam && d.kind != CM_KIND_NIIR) return 0;
    const cm_filter &fpre = d.filters[qam ? QF_PRE_LP : NF_PRE_LP];       // slot 9 = QF_ENC_PRE = NF_ENC_PRE
    if (!fpre.nsec || fpre.rate > 1) return 0;
    static const int th[3] = {1, 2, 2}, lpre[3] = {23, 23, 31}, wmax[3] = {768, 1536, 2048};
    for (int k = 0; k < 3; ++k) {
        if (d.width > wmax[k] || fpre.n + fpre.shift > 32 * th[k] * lpre[k]) continue;
        build_filter_L(fpre, fh[9], tab, lpre[k], 1, 32 * th[k]);
        return k + 1;
    }
    return 0;
}

static int plan_row_kernel(const cm_desc &d, FiltHdr *fh, std::vector<double> &tab) {
    if (d.kind == CM_KIND_QAM_BANDSPLIT) {           // k_qam_bs_row2: one chunk length for its three 2x use-sites
        const cm_filter &fbp = d.filters[QF_BP2X], &fbs = d.filters[QF_BS2X], &flp = d.filters[QF_DEMOD_LP];
        if (!fbp.nsec || !fbs.nsec || !flp.nsec) return 0;
        static const int th[3] = {1, 2, 2}, la[3] = {46, 46, 62}, lb[3] = {50, 50, 66};
        int need = fbp.n + fbp.shift;
        if (fbs.n + fbs.shift > need) need = fbs.n + fbs.shift;
        if (flp.n + flp.shift > need) need = flp.n + flp.shift;
        for (int k = 0; k < 3; ++k) {
            const int ll = need <= 32 * th[k] * la[k] ? la[k] : (need <= 32 * th[k] * lb[k] ? lb[k] : 0);
            if (!ll) continue;
            build_filter_L(fbp, fh[6], tab, ll, 1, 32 * th[k]);
            build_filter_L(flp, fh[7], tab, ll, 1, 32 * th[k]);
            build_filter_L(fbs, fh[8], tab, ll, 1, 32 * th[k]);
            return k + 1;
        }
        return 0;
    }
    if (d.kind < CM_KIND_NTSC_COMB || d.kind > CM_KIND_PAL_3D) return 0;
    const bool pald = d.kind == CM_KIND_PAL_D ||
                      (d.kind == CM_KIND_PAL_3D && !(d.flags & (CM_FLAG_PAL3D_SIN | CM_FLAG_PAL3D_COS)));
    const cm_filter &fbp = d.filters[QF_BP2X], &flp = d.filters[pald ? QF_PALD_LP : QF_DEMOD_LP], &fpre = d.filters[QF_PRE_LP];
    if (!fbp.nsec || !flp.nsec || !fpre.nsec) return 0;
    static const int nws[3] = {2, 4, 4};            // RowL<1..3> of cm_qam.cuh
    static const int lbp[3] = {26, 26, 34}, lpa[3] = {46, 46, 62}, lpb[3] = {50, 50, 66}, lpre[3] = {23, 23, 31};
    for (int k = 0; k < 3; ++k) {
        const int nw = nws[k], th = nw / 2;
        if (fbp.n + fbp.shift > 32 * nw * lbp[k]) continue;
        if (fpre.n + fpre.shift > 32 * th * lpre[k]) continue;
        int ll = 0;
        if (flp.n + flp.shift <= 32 * th * lpa[k]) ll = lpa[k];
        else if (flp.n + flp.shift <= 32 * th * lpb[k]) ll = lpb[k];
        if (!ll) continue;
        build_filter_L(fbp, fh[6], tab, lbp[k], 1, 32 * nw);
        build_filter_L(flp, fh[7], tab, ll, 1, 32 * th);
        build_filter_L(fpre, fh[8], tab, lpre[k], 1, 32 * th);
        return k + 1;
    }
    return 0;
}

// Geometry of k_secam_decode2 (cm_secam.cuh: SecGeo) for this line length: 1 = 2 warps, 3 = 4 warps; fills the SF_ROW_*
// headers and section tables.  0: none fits (the multi-row kernel serves the line).
static int plan_secam_kernel(const cm_desc &d, FiltHdr *fh, std::vector<double> &tab) {
    if (d.kind != CM_KIND_SECAM) return 0;
    static const int geo[2] = {1, 3}, th[2] = {1, 2}, l1[2] = {25, 33}, l2[2] = {50, 66}, iter[2] = {12, 16};
    static const int src[5] = {SF_LUMA_BS, SF_CHROMA_BP, SF_ANTI_BELL, SF_FM_LP, SF_DE_EMPH};
    const int ncc4 = (d.width + d.width / 40 - 1 + 3) & ~3;
    for (int k = 0; k < 2; ++k) {
        bool ok = ncc4 <= 32 * 2 * th[k] * iter[k] && d.width <= 16 * 32 * 2 * th[k];
        for (int i = 0; i < 5 && ok; ++i) {
            const cm_filter &f = d.filters[src[i]];
            if (!f.nsec) continue;
            const int cap = 32 * th[k] * (f.rate == 2 ? l2[k] : l1[k]);
            if (f.rate > 2 || f.n + f.shift > cap) ok = false;
        }
        if (!ok || !d.filters[SF_LUMA_BS].nsec || !d.filters[SF_CHROMA_BP].nsec || !d.filters[SF_FM_LP].nsec) continue;
        for (int i = 0; i < 5; ++i) {
            const cm_filter &f = d.filters[src[i]];
            if (f.nsec) build_filter_L(f, fh[7 + i], tab, f.rate == 2 ? l2[k] : l1[k], 1, 32 * th[k]);
        }
        // the row encoder (k_secam_encode_row2): chroma low-pass and LF pre-emphasis sites, same team geometry
        const cm_filter &fp = d.filters[SF_PRE_LP], &fe = d.filters[SF_PRE_EMPH];
        const int lf[2] = {13, 15}, le[2] = {13, 17}, lanes = 32 * 2 * th[k];      // (SecEncGeo: all warps as one team)
        if (fp.nsec && fp.n + fp.shift <= lanes * le[k] && (!fe.nsec || fe.n + fe.shift <= lanes * le[k]) &&
            d.width <= lanes * lf[k]) {
            build_filter_L(fp, fh[12], tab, le[k], 1, lanes);
            if (fe.nsec) build_filter_L(fe, fh[13], tab, le[k], 1, lanes);
        }
        return geo[k];
    }
    return 0;
}

// Geometry of k_niir_decode2 (cm_niir.cuh: NiirGeo): 1 = 2 warps x 39 samples per lane, 3 = 4 warps x 51; fills NF_ROW_*.
static int plan_niir_kernel(const cm_desc &d, FiltHdr *fh, std::vector<double> &tab) {
    if (d.kind != CM_KIND_NIIR) return 0;
    const cm_filter &fbp = d.filters[NF_UP_BP], &flp = d.filters[NF_BASE_LP];
    if (!fbp.nsec || !flp.nsec || fbp.rate != 3 || flp.rate != 3) return 0;
    static const int geo[2] = {1, 3}, nw[2] = {2, 4}, l3[2] = {39, 51};
    for (int k = 0; k < 2; ++k) {
        const int cap = 32 * nw[k] * l3[k];
        if (fbp.n + fbp.shift > cap || flp.n + flp.shift > cap) continue;
        build_filter_L(fbp, fh[4], tab, l3[k], 1, 32 * nw[k]);
        build_filter_L(flp, fh[5], tab, l3[k], 1, 32 * nw[k]);
        return geo[k];
    }
    return 0;
}

// Geometry of k_proto_decode2 / k_proto_encode_row2 (cm_proto.cuh: ProtoGeo): 1 = 4 warps, 3 = 8 warps; fills PF_ROW_* / PF_ENC_PRE.
static int plan_proto_kernel(const cm_desc &d, FiltHdr *fh, std::vector<double> &tab) {
    if (d.kind != CM_KIND_PROTOSECAM) return 0;
    const cm_filter &fbp = d.filters[PF_BP_UP], &fbs = d.filters[PF_BS_UP], &fpost = d.filters[PF_POST_LP],
                    &fpre = d.filters[PF_PRE_LP];
    if (!fbp.nsec || !fbs.nsec || !fpost.nsec || !fpre.nsec) return 0;
    static const int geo[2] = {1, 3}, th[2] = {2, 4}, l3[2] = {39, 51}, l1[2] = {13, 17};
    for (int k = 0; k < 2; ++k) {
        const int cap3 = 32 * th[k] * l3[k], cap1 = 32 * th[k] * l1[k];
        if (fbp.n + fbp.shift > cap3 || fbs.n + fbs.shift > cap3 || fpost.n + fpost.shift > cap3 || fpre.n + fpre.shift > cap1 ||
            d.width > 16 * 32 * 2 * th[k] / 2)
            continue;
        build_filter_L(fbp, fh[4], tab, l3[k], 1, 32 * th[k]);
        build_filter_L(fbs, fh[5], tab, l3[k], 1, 32 * th[k]);
        build_filter_L(fpost, fh[6], tab, l3[k], 1, 32 * th[k]);
        build_filter_L(fpre, fh[7], tab, l1[k], 1, 32 * th[k]);
        return geo[k];
    }
    return 0;
}

// Row-independent carrier of k_qam_rows2 / k_secam_decode2: sin / cos of (j * step) for the 2x sample index j, tail
// replicated, in the load order of LoadPoly2Carrier: [task][i / 2][chunk][i & 1] with j = chunk * L + i.
static void build_carrier_table(unsigned long long step, const FiltHdr &fl, int th, std::vector<double> &out) {
    const int L = fl.L, nchunks = 32 * th;
    out.assign((size_t)2 * fl.npad, 0.0);
    for (int chunk = 0; chunk < nchunks; ++chunk)
        for (int i = 0; i < L; ++i) {
            int j = chunk * L + i;
            if (j > fl.n - 1) j = fl.n - 1;
            const unsigned long long ph = (unsigned long long)j * step;                // wraps mod one turn
            const double turns = (double)(long long)ph * 5.421010862427522170e-20;     // 2^-64: [-0.5, 0.5)
            const size_t at = 2 * ((size_t)(i >> 1) * nchunks + chunk) + (i & 1);
            out[at] = sin(6.283185307179586476925 * turns);
            out[(size_t)fl.npad + at] = cos(6.283185307179586476925 * turns);
        }
}

// Aligned polyphase form of a rational resampler (PolyHdr, cm_common.cuh).  scipy.signal.resample_poly / upfirdn
// (SURVEY.md section 8 a9): y[j] = sum_i h[c - i up] x[i], c = half + j down, taps 0 .. 2 half, zeros outside the line.
// For j = up m + r:  c = up (m down) + (half + r down), so the lowest line index is m down + lo_r with
// lo_r = ceil((r down - half) / up) and the tap that meets it is t_r = half + r down - lo_r up  (2 half - up < t_r <= 2 half).
// Window of group m: starts at s = (m down + lo_0 + FP) & ~3; phase r begins d_r = a + lo_r - lo_0 samples into it.
static bool build_poly(const cm_resampler &rs, PolyHdr &ph, std::vector<double> &tab) {
    memset(&ph, 0, sizeof(ph));
    if (rs.ntaps == 0 || rs.up > 4) return false;
    auto ceil_div = [](int a, int b) { return a >= 0 ? (a + b - 1) / b : -((-a) / b); };
    int K = 0, lo[4] = {0, 0, 0, 0}, t_r[4] = {0, 0, 0, 0};
    for (int r = 0; r < rs.up; ++r) {
        lo[r] = ceil_div(r * rs.down - rs.half, rs.up);
        t_r[r] = rs.half + r * rs.down - lo[r] * rs.up;
        const int k = t_r[r] / rs.up + 1 + (lo[r] - lo[0]);        // reach of phase r inside the window (a = 0)
        if (k > K) K = k;
    }
    ph.up = rs.up;
    ph.down = rs.down;
    ph.lo0 = lo[0];
    ph.KU = (K + 3 + 7) & ~7;
    ph.stride = ph.KU;
    if (((ph.stride >> 2) & 1) == 0) ph.stride += 4;          // stride / 4 odd: rows read together sit on distinct banks
    ph.FP = (-lo[0] + 3) & ~3;
    if (ph.FP < 0) ph.FP = 0;
    ph.off = (int)tab.size();
    tab.resize(tab.size() + (size_t)4 * rs.up * ph.stride, 0.0);
    for (int a = 0; a < 4; ++a)
        for (int r = 0; r < rs.up; ++r)
            for (int q = 0; q < ph.KU; ++q) {
                const int t = t_r[r] + (a + lo[r] - lo[0] - q) * rs.up;
                if (t >= 0 && t <= 2 * rs.half) tab[(size_t)ph.off + (size_t)(a * rs.up + r) * ph.stride + q] = rs.taps[t];
            }
    return true;
}

template <typename T>
static void fill_params(const cm_desc &d, DevParams<T> &p, const FiltHdr *fh, const ResHdr *rh, const void *tab,
                        const void *taps) {
    memset(&p, 0, sizeof(p));
    p.kind = d.kind;
    p.flags = d.flags;
    p.W = d.width;
    p.H = d.height;
    p.Wc = d.comp_width;
    p.Wo = d.out_width;
    p.digital_shift = d.digital_shift;
    p.odd_first = d.odd_first;
    p.even_first = d.even_first;
    p.ref_line = d.ref_line;
    p.frame_cycle = d.frame_cycle;
    p.frame_shift = d.frame_shift_turns;
    p.line_shift = d.line_shift_turns;
    for (int i = 0; i < CM_NPHASE; ++i) p.phases[i] = d.phases[i];
    for (int i = 0; i < CM_NSCAL; ++i) p.scalars[i] = (T)d.scalars[i];
    for (int i = 0; i < 9; ++i) { p.enc[i] = (T)d.enc_matrix[i]; p.dec[i] = (T)d.dec_matrix[i]; p.encd[i] = d.enc_matrix[i]; }
    p.ident_enc = p.ident_dec = 1;
    for (int i = 0; i < 9; ++i) {
        const double id = (i % 4 == 0) ? 1.0 : 0.0;
        if (d.enc_matrix[i] != id) p.ident_enc = 0;
        if (d.dec_matrix[i] != id) p.ident_dec = 0;
    }
    for (int i = 0; i < CM_NFILT; ++i) p.filt[i] = fh[i];
    // line-buffer geometry: every buffer that feeds an IIR is padded to the site's 32*L*nsuper
    auto up4 = [](int v) { return (v + 3) & ~3; };
    int n1p = up4(d.width > d.comp_width ? d.width : d.comp_width), n2p = 2 * up4(d.comp_width),
        n3p = 3 * up4(d.comp_width);
    for (int i = 0; i < CM_NFILT; ++i) {
        if (!fh[i].nsec) continue;
        if (fh[i].rate == 1 && fh[i].npad > n1p) n1p = fh[i].npad;
        if (fh[i].rate == 2 && fh[i].npad > n2p) n2p = fh[i].npad;
        if (fh[i].rate == 3 && fh[i].npad > n3p) n3p = fh[i].npad;
    }
    p.n1p = up4(n1p);
    p.hb2 = up4((n2p + 1) / 2);
    if (d.kind <= CM_KIND_PAL_3D && p.hb2 < p.n1p) p.hb2 = p.n1p;   // QAM kernels park two 1x rows in one 2x buffer
    p.hb3 = up4((n3p + 2) / 3);
    for (int i = 0; i < CM_NRES; ++i) p.res[i] = rh[i];
    p.tab = (const T *)tab;
    p.taps = (const T *)taps;
    for (int r = 0; r < 2; ++r)
        if (d.resamplers[r].ntaps > 0 && d.resamplers[r].ntaps <= 64)
            for (int i = 0; i < d.resamplers[r].ntaps; ++i) {
                p.firc[r][i] = (T)d.resamplers[r].taps[i];
                p.fircp[r][i][0] = p.fircp[r][i][1] = (float)d.resamplers[r].taps[i];
            }
}

template <typename T>
static int upload(const std::vector<double> &src, void **dst) {
    std::vector<T> tmp(src.size() ? src.size() : 1);
    for (size_t i = 0; i < src.size(); ++i) tmp[i] = (T)src[i];
    CUDA_TRY(cudaMalloc(dst, tmp.size() * sizeof(T)));
    CUDA_TRY(cudaMemcpy(*dst, tmp.data(), tmp.size() * sizeof(T), cudaMemcpyHostToDevice));
    return CM_OK;
}

// ------------------------------------------------------------------------------------------------------------
// PAL-D as a banded matrix product (cm_pald_mma.cu)
// ------------------------------------------------------------------------------------------------------------
// resample_poly of one line: out[j] = sum_i x[i] taps[half + j down - i up], zeros outside the line
static void resample_line(const std::vector<double> &x, const cm_resampler &rs, std::vector<double> &out) {
    const int n = (int)x.size(), nout = (n * rs.up + rs.down - 1) / rs.down;
    out.assign(nout, 0.0);
    for (int j = 0; j < nout; ++j) {
        const int c = rs.half + j * rs.down;
        const int lo = c - 2 * rs.half <= 0 ? 0 : (c - 2 * rs.half + rs.up - 1) / rs.up;
        const int hi = c / rs.up < n - 1 ? c / rs.up : n - 1;
        double acc = 0.0;
        for (int i = lo; i <= hi; ++i) acc += x[i] * rs.taps[c - i * rs.up];
        out[j] = acc;
    }
}

// one IIR use-site on one line: `shift` copies of the last sample appended, second-order sections (DF-II-T, zero state),
// the first `shift` outputs dropped (oracle/dsp.py: Filt)
static void iir_line(std::vector<double> &x, const cm_filter &f) {
    const size_t n = x.size();
    std::vector<double> y(x);
    y.resize(n + f.shift, x[n - 1]);
    for (int s = 0; s < f.nsec; ++s) {
        const double *c = f.sos[s];
        double z1 = 0.0, z2 = 0.0;
        for (double &v : y) {
            const double in = v, out = c[0] * in + z1;
            z1 = c[1] * in - c[3] * out + z2;
            z2 = c[2] * in - c[4] * out;
            v = out;
        }
    }
    for (size_t i = 0; i < n; ++i) x[i] = y[i + f.shift];
}

static bool pald_kind(const cm_desc &d) {
    return d.kind == CM_KIND_PAL_D || (d.kind == CM_KIND_PAL_3D && !(d.flags & (CM_FLAG_PAL3D_SIN | CM_FLAG_PAL3D_COS)));
}

// The linear map of pass 1 of the PAL-D decoder (k_qam_rows2<PALD> before the row's phase rotation), from the signal of
// the W composite samples to the planes of each sample x: M[i * 4W + 4x + plane], planes a', b', LPpre a', LPpre b'.
// Restated on unit impulses: up2, band-pass, down2, up2, the table carrier (sin for a', cos for b'), the AM low-pass,
// down2, then the encoder's chroma low-pass.
static void pald_matrix(const cm_desc &d, std::vector<double> &M) {
    const int W = d.width;
    const cm_resampler &up = d.resamplers[QR_UP2], &dn = d.resamplers[QR_DOWN2];
    const cm_filter &fbp = d.filters[QF_BP2X], &flp = d.filters[QF_PALD_LP], &fpre = d.filters[QF_PRE_LP];
    std::vector<double> car[2];
    car[0].resize(2 * W);
    car[1].resize(2 * W);
    for (int j = 0; j < 2 * W; ++j) {      // as build_carrier_table
        const unsigned long long ph = (unsigned long long)j * d.phases[QP_STEP2X];
        const double turns = (double)(long long)ph * 5.421010862427522170e-20;
        car[0][j] = sin(6.283185307179586476925 * turns);
        car[1][j] = cos(6.283185307179586476925 * turns);
    }
    M.assign((size_t)W * 4 * W, 0.0);
    std::vector<double> x(W), g, c, g2, pr(2 * W), a;
    for (int i = 0; i < W; ++i) {
        std::fill(x.begin(), x.end(), 0.0);
        x[i] = 1.0;
        resample_line(x, up, g);
        iir_line(g, fbp);
        resample_line(g, dn, c);
        resample_line(c, up, g2);
        for (int t = 0; t < 2; ++t) {
            for (int j = 0; j < 2 * W; ++j) pr[j] = g2[j] * car[t][j];
            iir_line(pr, flp);
            resample_line(pr, dn, a);
            double *row = &M[(size_t)i * 4 * W];
            for (int s = 0; s < W; ++s) row[4 * s + t] = a[s];
            iir_line(a, fpre);
            for (int s = 0; s < W; ++s) row[4 * s + 2 + t] = a[s];
        }
    }
}

// Reach of M (pald_matrix) around the diagonal: output sample x depends on the inputs [x - lo, x + hi], to 2^-26 of the
// largest coefficient of its plane.
static void pald_band(const std::vector<double> &M, int W, int &lo, int &hi) {
    double mx[4] = {0, 0, 0, 0};
    for (size_t k = 0; k < M.size(); ++k) mx[k & 3] = fmax(mx[k & 3], fabs(M[k]));
    lo = hi = 0;
    for (int i = 0; i < W; ++i)
        for (int n = 0; n < 4 * W; ++n)
            if (fabs(M[(size_t)i * 4 * W + n]) > ldexp(mx[n & 3], -26)) {
                const int x = n >> 2;
                if (x - i > lo) lo = x - i;
                if (i - x > hi) hi = i - x;
            }
}

// B operand of k_pald_mma (cm_host.h: PaldMmaArgs) for a float32 PAL-D handle whose band fits the compiled window; leaves
// the handle without it (the two-pass kernels serve it) otherwise.  The level map is folded in: the composite signal is
// (5 u / 255 - 1) / 3 for the byte u, so the planes are u . (5 / 765) M - (1 / 3) colsum(M).  Each column is scaled by a
// power of two (largest coefficient near 1000) and split into FP16 hi + lo.
static int plan_pald_mma(cm_modem *m) {
    const cm_desc &d = m->desc;
    const int W = d.width;
    if (m->precision != CM_FP32 || !m->tune.pald_mma || m->tune.onepass || m->tune.rows_v1 || !pald_kind(d) ||
        !m->pf.row_geo || d.comp_width != W || d.out_width != W || d.resamplers[QR_UP2].ntaps <= 0 ||
        d.resamplers[QR_DOWN2].ntaps <= 0)
        return CM_OK;
    std::vector<double> M;
    pald_matrix(d, M);
    int lo = 0, hi = 0;
    pald_band(M, W, lo, hi);
    if (lo > CM_PALD_KPRE || hi > CM_PALD_KW - CM_PALD_KPRE - CM_PALD_TS) return CM_OK;
    const int ntiles = (W + CM_PALD_TS - 1) / CM_PALD_TS, kc = CM_PALD_KW / 8, N = CM_PALD_N;
    std::vector<uint16_t> B((size_t)ntiles * 2 * CM_PALD_KW * N, 0);
    std::vector<float> cs((size_t)ntiles * 2 * N, 0.0f);
    for (int tile = 0; tile < ntiles; ++tile) {
        const int xs = tile * CM_PALD_TS - CM_PALD_KPRE;
        for (int n = 0; n < N; ++n) {
            const int x = tile * CM_PALD_TS + (n >> 2), col = 4 * x + (n & 3);
            float *inv = &cs[(size_t)tile * 2 * N + n], *bias = inv + N;
            *inv = 1.0f;
            if (x >= W) continue;
            double mx = 0.0, sum = 0.0;
            for (int i = 0; i < W; ++i) sum += M[(size_t)i * 4 * W + col];
            for (int k = 0; k < CM_PALD_KW; ++k)
                if (xs + k >= 0 && xs + k < W) mx = fmax(mx, fabs(M[(size_t)(xs + k) * 4 * W + col]) * (5.0 / 765.0));
            const double scale = mx > 0.0 ? ldexp(1.0, (int)floor(log2(1000.0 / mx))) : 1.0;
            *inv = (float)(1.0 / scale);
            *bias = (float)(-sum / 3.0);
            for (int k = 0; k < CM_PALD_KW; ++k) {
                if (xs + k < 0 || xs + k >= W) continue;
                const double r = M[(size_t)(xs + k) * 4 * W + col] * (5.0 / 765.0) * scale;
                const __half h = __float2half_rn((float)r);
                const __half l = __float2half_rn((float)(r - (double)__half2float(h)));
                const size_t at = ((size_t)(tile * 2) * kc + k / 8) * N * 8 + (size_t)n * 8 + (k & 7);
                B[at] = __half_as_ushort(h);
                B[at + (size_t)kc * N * 8] = __half_as_ushort(l);
            }
        }
    }
    CUDA_TRY(cudaMalloc(&m->d_mma_b, B.size() * sizeof(uint16_t)));
    CUDA_TRY(cudaMemcpy(m->d_mma_b, B.data(), B.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMalloc(&m->d_mma_cs, cs.size() * sizeof(float)));
    CUDA_TRY(cudaMemcpy(m->d_mma_cs, cs.data(), cs.size() * sizeof(float), cudaMemcpyHostToDevice));
    return CM_OK;
}

// Test hook: the matrix of pald_matrix (W x 4W, float64, row-major) and its band (lo, hi) for a PAL-D handle.
extern "C" int cm_pald_matrix(const cm_modem *m, double *out, int *band) {
    if (!m || !pald_kind(m->desc)) return fail(CM_ERR_UNSUPPORTED, "not a PAL-D handle%s");
    std::vector<double> M;
    pald_matrix(m->desc, M);
    if (out) memcpy(out, M.data(), M.size() * sizeof(double));
    if (band) pald_band(M, m->desc.width, band[0], band[1]);
    return CM_OK;
}

extern "C" int cm_abi_version(void) { return CM_ABI_VERSION; }
extern "C" int cm_sizeof_desc(void) { return (int)sizeof(cm_desc); }
extern "C" const char *cm_last_error(void) { return g_err; }
extern "C" int64_t cm_launch_count(void) { return g_launches.load(); }

extern "C" int cm_device_info(int *sm_count, int *cc_major, int *cc_minor) {
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return CM_OK;
}

extern "C" int cm_create(const cm_desc *desc, int precision, cm_modem **out) {
    if (!desc || !out) return fail(CM_ERR_INVALID, "null argument%s");
    if (desc->abi_version != CM_ABI_VERSION) return fail(CM_ERR_INVALID, "cm_desc.abi_version mismatch%s");
    if (precision != CM_FP32 && precision != CM_FP64) return fail(CM_ERR_INVALID, "bad precision%s");
    if (desc->width <= 0 || desc->height <= 0 || desc->comp_width <= 0 || desc->out_width <= 0)
        return fail(CM_ERR_INVALID, "bad raster size%s");
    if (desc->nfilters < 0 || desc->nfilters > CM_MAX_FILTERS || desc->nresamplers < 0 ||
        desc->nresamplers > CM_MAX_RESAMPLERS)
        return fail(CM_ERR_INVALID, "bad filter / resampler count%s");
    if (desc->frame_cycle <= 0) return fail(CM_ERR_INVALID, "frame_cycle must be positive%s");
    if ((desc->width & 3) || (desc->comp_width & 3) || (desc->out_width & 3))
        return fail(CM_ERR_UNSUPPORTED, "line widths must be multiples of 4 samples%s");
    switch (desc->kind) {
        case CM_KIND_QAM_BANDSPLIT:
        case CM_KIND_NTSC_COMB:
        case CM_KIND_NTSC_3D:
        case CM_KIND_PAL_D:
        case CM_KIND_PAL_3D:
        case CM_KIND_SECAM:
        case CM_KIND_NIIR:
        case CM_KIND_PROTOSECAM:
        case CM_KIND_MAC:
            break;
        default:
            return fail(CM_ERR_UNSUPPORTED, "modem kind not built%s");
    }
    if (desc->kind == CM_KIND_NTSC_3D && (desc->flags & CM_FLAG_NTSC_NO_COMB))
        // comb.py:96-109 over ntsc.py:71-72 averages the band-split chroma of two lines there; the fused 3-line kernel
        // does not (the Python mirror serves that composition through the composed path)
        return fail(CM_ERR_UNSUPPORTED, "Simple3DCombModem(NtscCombModem) without a usable line comb is not a fused kind%s");
    cm_modem *m = new (std::nothrow) cm_modem();
    if (!m) return fail(CM_ERR_NOMEM, "out of host memory%s");
    m->desc = *desc;
    m->precision = precision;
    {   // tuning knobs: the environment is read here, once per handle (cm_host.h: cm_tune)
        auto env_int = [](const char *name, int dflt) {
            const char *e = getenv(name);
            if (!e) return dflt;
            const int v = atoi(e);
            return v > 0 ? v : dflt;
        };
        m->tune.onepass = getenv("CM_ONEPASS") != nullptr;
        m->tune.rows_v1 = getenv("CM_ROWS_V1") != nullptr;
        m->tune.rpc = env_int("CM_RPC", m->tune.rpc);
        m->tune.chunk = env_int("CM_CHUNK", m->tune.chunk);
        m->tune.host_chunk = env_int("CM_HOST_CHUNK", m->tune.host_chunk);
        if (const char *e = getenv("CM_HOST_ROLES")) m->tune.host_roles = atoi(e);
        m->tune.rows_max = env_int("CM_ROWS_MAX", m->tune.rows_max);
        m->tune.min_warps = env_int("CM_MIN_WARPS", m->tune.min_warps);
        m->tune.mac_threads = env_int("CM_MAC_THREADS", m->tune.mac_threads) & ~31;
        if (m->tune.mac_threads < 32) m->tune.mac_threads = 32;
        if (m->tune.mac_threads > CM_NTHREADS) m->tune.mac_threads = CM_NTHREADS;       // the kernels' launch bound
        if (const char *e = getenv("CM_OVERLAP")) m->tune.overlap = atoi(e);
        if (const char *e = getenv("CM_PALD_MMA")) m->tune.pald_mma = atoi(e) != 0;
    }
    cudaError_t e = cudaGetDevice(&m->device);
    if (e != cudaSuccess) { delete m; return fail(CM_ERR_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e)); }
    cudaDeviceGetAttribute(&m->sm_count, cudaDevAttrMultiProcessorCount, m->device);
    cudaDeviceGetAttribute(&m->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, m->device);

    FiltHdr fh[CM_NFILT];
    ResHdr rh[CM_NRES];
    memset(fh, 0, sizeof(fh));
    memset(rh, 0, sizeof(rh));
    std::vector<double> tab, taps;
    for (int i = 0; i < desc->nfilters; ++i) {
        const cm_filter &f = desc->filters[i];
        if (f.nsec == 0) continue;
        if (f.nsec < 0 || f.nsec > CM_MAX_SECTIONS || f.shift < 0 || f.n <= 0 || f.rate < 1 || f.rate > 3) {
            delete m;
            return fail(CM_ERR_INVALID, "bad cm_filter%s");
        }
        build_filter(f, fh[i], tab);
    }
    for (int i = 0; i < desc->nresamplers; ++i) {
        const cm_resampler &r = desc->resamplers[i];
        if (r.ntaps == 0) continue;
        if (r.ntaps < 0 || r.ntaps > CM_MAX_TAPS || r.up <= 0 || r.down <= 0 || r.ntaps != 2 * r.half + 1) {
            delete m;
            return fail(CM_ERR_INVALID, "bad cm_resampler%s");
        }
        rh[i].up = r.up;
        rh[i].down = r.down;
        rh[i].half = r.half;
        rh[i].ntaps = r.ntaps;
        rh[i].off = (int)taps.size();
        taps.insert(taps.end(), r.taps, r.taps + r.ntaps);
    }
    std::vector<double> ptab;
    PolyHdr poly[CM_NRES];
    memset(poly, 0, sizeof(poly));
    int mac_fp = 0, mac_bp = 0;
    if (desc->kind == CM_KIND_MAC)
        for (int i = 0; i < desc->nresamplers && i < CM_NRES; ++i)
            if (build_poly(desc->resamplers[i], poly[i], ptab)) {
                if (poly[i].FP > mac_fp) mac_fp = poly[i].FP;
                if (poly[i].KU > mac_bp) mac_bp = poly[i].KU;
            }
    mac_fp = (mac_fp + 31) & ~31;          // one front pad for every resampler, a whole number of 32-element skew blocks
    int mac_skew = 0;
    for (int i = 0; i < CM_NRES; ++i)
        if (poly[i].up && poly[i].down % 8 == 0) mac_skew = -1;
    for (int i = 0; i < CM_NRES; ++i)
        if (poly[i].up) { poly[i].FP = mac_fp; poly[i].skew = mac_skew; }
    ptab.resize((ptab.size() + 3) & ~(size_t)3, 0.0);
    memset(&m->mcf, 0, sizeof(m->mcf));
    memset(&m->mcd, 0, sizeof(m->mcd));
    if (desc->kind == CM_KIND_MAC && !getenv("CM_MAC_SMEM_TAPS")) {       // (the environment switch is the A/B hook)
        // constant-bank copies of the tables whose shape matches a compiled one (MacConst, cm_common.cuh): row (a * up + r) of
        // the polyphase table of a slot holds the taps of phase r for window alignment a (build_poly)
        auto fill = [&](const PolyHdr &ph, int a, int r, auto *dstf, auto *dstd, int ku) {
            for (int q = 0; q < ku; ++q) {
                const double v = q < ph.KU ? ptab[(size_t)ph.off + (size_t)(a * ph.up + r) * ph.stride + q] : 0.0;
                dstf[q] = (float)v;
                dstd[q] = v;
            }
        };
        const PolyHdr &pl = poly[MR_LUMA_IN], &pc = poly[MR_CHROMA_IN], &po = poly[MR_OUT], &pi = poly[MR_COMP_IN];
        if (pl.up == 3 && pl.down % 4 == 0 && pl.KU <= MacShape::KL) {
            const int a = (pl.lo0 + pl.FP) & 3;
            for (int r = 0; r < 3; ++r) fill(pl, a, r, m->mcf.luma[r], m->mcd.luma[r], MacShape::KL);
            m->mcf.ok_luma = m->mcd.ok_luma = 1;
            if (mac_bp < MacShape::KL) mac_bp = MacShape::KL;       // the unrolled loop reads the whole compiled window
        }
        if (pc.up == 3 && pc.down % 4 == 0 && pc.KU <= MacShape::KC) {
            const int a = (pc.lo0 + pc.FP) & 3;
            for (int r = 0; r < 3; ++r) fill(pc, a, r, m->mcf.chroma[r], m->mcd.chroma[r], MacShape::KC);
            m->mcf.ok_chroma = m->mcd.ok_chroma = 1;
            if (mac_bp < MacShape::KC) mac_bp = MacShape::KC;
        }
        if (po.up == 2 && po.KU <= MacShape::KO) {
            for (int j = 0; j < 4; ++j) {
                const int a = (po.down * j + po.lo0 + po.FP) & 3;
                for (int r = 0; r < 2; ++r) fill(po, a, r, m->mcf.out[j][r], m->mcd.out[j][r], MacShape::KO);
            }
            m->mcf.ok_out = m->mcd.ok_out = 1;
            if (mac_bp < MacShape::KO) mac_bp = MacShape::KO;
        }
        if (pi.up == 3 && pi.KU <= MacShape::KI) {
            for (int j = 0; j < 4; ++j) {
                const int a = (pi.down * j + pi.lo0 + pi.FP) & 3;
                for (int r = 0; r < 3; ++r) fill(pi, a, r, m->mcf.comp[j][r], m->mcd.comp[j][r], MacShape::KI);
            }
            m->mcf.ok_comp = m->mcd.ok_comp = 1;
            if (mac_bp < MacShape::KI) mac_bp = MacShape::KI;
        }
    }
    const int row_geo = plan_row_kernel(*desc, fh, tab);
    const int enc_geo = plan_encode_kernel(*desc, fh, tab);
    std::vector<double> ctab;
    if (row_geo) build_carrier_table(desc->phases[QP_STEP2X], fh[7], row_geo == 1 ? 1 : 2, ctab);
    const int sec_geo = plan_secam_kernel(*desc, fh, tab);
    if (sec_geo) build_carrier_table(desc->phases[SP_FM_STEP2X], fh[10], sec_geo == 1 ? 1 : 2, ctab);
    int niir_geo = plan_niir_kernel(*desc, fh, tab);
    if (!niir_geo) niir_geo = plan_proto_kernel(*desc, fh, tab);
    int rc;
    if (precision == CM_FP32) {
        rc = upload<float>(tab, &m->d_tab);
        if (rc == CM_OK) rc = upload<float>(taps, &m->d_taps);
        if (rc == CM_OK) rc = upload<float>(ctab, &m->d_ctab);
        if (rc == CM_OK) rc = upload<float>(ptab, &m->d_ptab);
        fill_params<float>(*desc, m->pf, fh, rh, m->d_tab, m->d_taps);
        m->pf.ptab = (const float *)m->d_ptab;
        memcpy(m->pf.poly, poly, sizeof(poly));
        m->pf.mac_fp = mac_fp;
        m->pf.mac_skew = mac_skew;
        m->pf.mac_bp = mac_bp;
        m->pf.ctab = (const float *)m->d_ctab;
        m->pf.row_geo = row_geo ? row_geo : (sec_geo ? sec_geo : niir_geo);
        m->pf.enc_geo = enc_geo;
        if (rc == CM_OK) rc = plan_pald_mma(m);
    } else {
        rc = upload<double>(tab, &m->d_tab);
        if (rc == CM_OK) rc = upload<double>(taps, &m->d_taps);
        if (rc == CM_OK) rc = upload<double>(ctab, &m->d_ctab);
        if (rc == CM_OK) rc = upload<double>(ptab, &m->d_ptab);
        fill_params<double>(*desc, m->pd, fh, rh, m->d_tab, m->d_taps);
        m->pd.ptab = (const double *)m->d_ptab;
        memcpy(m->pd.poly, poly, sizeof(poly));
        m->pd.mac_fp = mac_fp;
        m->pd.mac_skew = mac_skew;
        m->pd.mac_bp = mac_bp;
        m->pd.ctab = (const double *)m->d_ctab;
        m->pd.row_geo = row_geo ? row_geo : (sec_geo ? sec_geo : niir_geo);
        m->pd.enc_geo = enc_geo;
    }
    if (rc != CM_OK) { cm_destroy(m); return rc; }
    *out = m;
    return CM_OK;
}

extern "C" void cm_destroy(cm_modem *m) {
    if (!m) return;
    cudaFree(m->d_tab);
    cudaFree(m->d_taps);
    cudaFree(m->d_ctab);
    cudaFree(m->d_ptab);
    cudaFree(m->d_mma_b);
    cudaFree(m->d_mma_cs);
    if (m->last_use) cudaEventDestroy(m->last_use);
    if (m->s2) cudaStreamDestroy(m->s2);
    for (int i = 0; i < 2; ++i) {
        if (m->ev_p1[i]) cudaEventDestroy(m->ev_p1[i]);
        if (m->ev_p2[i]) cudaEventDestroy(m->ev_p2[i]);
    }
    for (int i = 0; i < cm_modem::kHostBufs; ++i) {
        cudaFree(m->d_in[i]);
        cudaFree(m->d_out[i]);
        cudaFree(m->d_mid[i]);
        cudaFree(m->d_rgb[i]);
        if (m->ev_in[i]) cudaEventDestroy(m->ev_in[i]);
        if (m->ev_k[i]) cudaEventDestroy(m->ev_k[i]);
        if (m->ev_mid[i]) cudaEventDestroy(m->ev_mid[i]);
        if (m->ev_out[i]) cudaEventDestroy(m->ev_out[i]);
    }
    for (int i = 0; i < cm_modem::kHostStreams; ++i) {
        if (m->hs[i]) cudaStreamDestroy(m->hs[i]);
    }
    for (int i = 0; i < 12; ++i) cudaFree(m->d_aux[i]);
    cm_timing_reset(m);
    delete m;
}

// ------------------------------------------------------------------------------------------------------------
// launches
// ------------------------------------------------------------------------------------------------------------
void *cm_ensure_aux(cm_modem *m, size_t bytes, int which) {
    const int k = which * 4 + m->aux_slot;
    if (m->aux_cap[k] >= bytes) return m->d_aux[k];
    // the old buffer may still be in use by kernels already queued on some stream
    if (cudaDeviceSynchronize() != cudaSuccess) { fail(CM_ERR_CUDA, "cudaDeviceSynchronize failed%s"); return nullptr; }
    cudaFree(m->d_aux[k]);
    m->d_aux[k] = nullptr;
    m->aux_cap[k] = 0;
    cudaError_t e = cudaMalloc(&m->d_aux[k], bytes);
    if (e != cudaSuccess) { fail(CM_ERR_NOMEM, "cudaMalloc(aux): %s", cudaGetErrorString(e)); return nullptr; }
    m->aux_cap[k] = bytes;
    return m->d_aux[k];
}

extern "C" int cm_timing_enable(cm_modem *m, int on) {
    if (!m) return fail(CM_ERR_INVALID, "null handle%s");
    m->timing = on != 0;
    return CM_OK;
}

extern "C" int cm_phase_profile(cm_modem *m, void *device_counters) {
    if (!m) return fail(CM_ERR_INVALID, "null handle%s");
    m->phase_prof = (unsigned long long *)device_counters;
    return CM_OK;
}

extern "C" int cm_timing_reset(cm_modem *m) {
    if (!m) return fail(CM_ERR_INVALID, "null handle%s");
    for (auto &e : m->events) { cudaEventDestroy(e.a); cudaEventDestroy(e.b); }
    m->events.clear();
    return CM_OK;
}

extern "C" int cm_timing_read(cm_modem *m, int id, double *total_ms, int64_t *launches) {
    if (!m) return fail(CM_ERR_INVALID, "null handle%s");
    double tot = 0.0;
    int64_t n = 0;
    for (auto &e : m->events) {
        if (e.id != id) continue;
        CUDA_TRY(cudaEventSynchronize(e.b));
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, e.a, e.b));
        tot += ms;
        ++n;
    }
    if (total_ms) *total_ms = tot;
    if (launches) *launches = n;
    return CM_OK;
}

template <typename T>
static int dispatch_encode(cm_modem *m, IoArgs<T> io, cudaStream_t st) {
    switch (m->desc.kind) {
        case CM_KIND_QAM_BANDSPLIT:
        case CM_KIND_NTSC_COMB:
        case CM_KIND_NTSC_3D:
        case CM_KIND_PAL_D:
        case CM_KIND_PAL_3D:
            return qam_encode<T>(m, io, st);
        case CM_KIND_SECAM:
            return secam_encode<T>(m, io, st);
        case CM_KIND_NIIR:
            return niir_encode<T>(m, io, st);
        case CM_KIND_PROTOSECAM:
            return proto_encode<T>(m, io, st);
        case CM_KIND_MAC:
            return mac_encode<T>(m, io, st);
        default:
            return fail(CM_ERR_UNSUPPORTED, "encode: modem kind not built%s");
    }
}

template <typename T>
static int dispatch_decode(cm_modem *m, IoArgs<T> io, int mode, cudaStream_t st) {
    const int kind = m->desc.kind;
    if (mode != CM_MODE_DEFAULT && (kind < CM_KIND_QAM_BANDSPLIT || kind > CM_KIND_PAL_3D))
        return fail(CM_ERR_INVALID, "cm_window.mode is only defined for the QAM family%s");
    if (mode < CM_MODE_DEFAULT || mode > CM_MODE_EXTRACT_CHROMA) return fail(CM_ERR_INVALID, "bad cm_window.mode%s");
    switch (kind) {
        case CM_KIND_QAM_BANDSPLIT:
        case CM_KIND_NTSC_COMB:
        case CM_KIND_NTSC_3D:
        case CM_KIND_PAL_D:
        case CM_KIND_PAL_3D:
            return qam_decode<T>(m, io, mode, st);
        case CM_KIND_SECAM:
            return secam_decode<T>(m, io, st);
        case CM_KIND_NIIR:
            return niir_decode<T>(m, io, st);
        case CM_KIND_PROTOSECAM:
            return proto_decode<T>(m, io, st);
        case CM_KIND_MAC:
            return mac_decode<T>(m, io, st);
        default:
            return fail(CM_ERR_UNSUPPORTED, "decode: modem kind not built%s");
    }
}

template <typename T>
static int run_ex(cm_modem *m, bool encode, const cm_window *win, const uint8_t *in_u8, const void *in_f,
                  uint8_t *out_u8, void *out_f, int64_t first_frame, int32_t nframes, void *stream) {
    if (!m) return fail(CM_ERR_INVALID, "null handle%s");
    if (nframes < 0 || first_frame < 0) return fail(CM_ERR_INVALID, "bad frame range%s");
    if (nframes == 0) return CM_OK;                    // an empty batch may come with null buffers
    if ((in_u8 == nullptr) == (in_f == nullptr)) return fail(CM_ERR_INVALID, "exactly one input buffer required%s");
    if (!out_u8 && !out_f) return fail(CM_ERR_INVALID, "no output buffer%s");
    // u8 frames move in 32-bit words, float frames in vectors of four samples (cm_fir.cuh: ld4 / st4; float4 for float)
    const uintptr_t falign = sizeof(T) == 4 ? 16 : alignof(T);
    if ((((uintptr_t)in_u8 | (uintptr_t)out_u8) & 3) || (((uintptr_t)in_f | (uintptr_t)out_f) & (falign - 1)))
        return fail(CM_ERR_INVALID, "misaligned frame buffer%s");
    IoArgs<T> io;
    memset(&io, 0, sizeof(io));
    io.in_u8 = in_u8;
    io.in_f = (const T *)in_f;
    io.out_u8 = out_u8;
    io.out_f = (T *)out_f;
    io.first_frame = first_frame;
    io.nframes = nframes;
    io.prof = m->phase_prof;
    if (win) {
        if (win->nrows <= 0 || win->out_begin < 0 || win->out_count < 0 || win->out_begin + win->out_count > win->nrows)
            return fail(CM_ERR_INVALID, "bad cm_window%s");
        io.nrows = win->nrows;
        io.y0 = win->y0;
        io.out_begin = win->out_begin;
        io.out_count = win->out_count;
    } else {
        io.nrows = m->desc.height;
        io.y0 = 0;
        io.out_begin = 0;
        io.out_count = m->desc.height;
    }
    CUDA_TRY(cudaSetDevice(m->device));
    const int mode = win ? win->mode : CM_MODE_DEFAULT;
    m->pf.phase0 = m->pd.phase0 = win ? win->phase_offset : 0ull;     // (a handle is not re-entrant)
    bool guard = m->aux_slot == 0;                // (the host entry points use their own scratch slot per stream)
    if (guard) {                                  // (a stream that is being captured into a CUDA graph is left alone)
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing((cudaStream_t)stream, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
            cudaGetLastError();
            guard = false;
        }
    }
    if (guard) {
        if (!m->last_use) CUDA_TRY(cudaEventCreateWithFlags(&m->last_use, cudaEventDisableTiming));
        if (m->used && m->last_stream != (cudaStream_t)stream) CUDA_TRY(cudaStreamWaitEvent((cudaStream_t)stream, m->last_use, 0));
    }
    // gridDim.z carries the frame index: at most 65535 frames per launch
    const size_t in_w = encode ? (size_t)m->desc.width * 3 : (size_t)m->desc.comp_width;
    const size_t out_w = encode ? (size_t)m->desc.comp_width : (size_t)m->desc.out_width * 3;
    for (int32_t base = 0; base < nframes; base += 65535) {
        IoArgs<T> part = io;
        part.nframes = nframes - base < 65535 ? nframes - base : 65535;
        part.first_frame = first_frame + base;
        const size_t in_off = (size_t)base * io.nrows * in_w, out_off = (size_t)base * io.nrows * out_w;
        if (part.in_u8) part.in_u8 += in_off;
        if (part.in_f) part.in_f += in_off;
        if (part.out_u8) part.out_u8 += out_off;
        if (part.out_f) part.out_f += out_off;
        int rc = encode ? dispatch_encode<T>(m, part, (cudaStream_t)stream)
                        : dispatch_decode<T>(m, part, mode, (cudaStream_t)stream);
        if (rc) return rc;
    }
    if (guard) {
        CUDA_TRY(cudaEventRecord(m->last_use, (cudaStream_t)stream));
        m->last_stream = (cudaStream_t)stream;
        m->used = true;
    }
    return CM_OK;
}

extern "C" int cm_encode_ex(cm_modem *m, const cm_window *win, const uint8_t *rgb_u8, const void *rgb_float,
                            uint8_t *comp_u8, void *comp_float, int64_t first_frame, int32_t nframes,
                            void *stream) {
    if (!m) return fail(CM_ERR_INVALID, "null handle%s");
    return m->precision == CM_FP32
               ? run_ex<float>(m, true, win, rgb_u8, rgb_float, comp_u8, comp_float, first_frame, nframes, stream)
               : run_ex<double>(m, true, win, rgb_u8, rgb_float, comp_u8, comp_float, first_frame, nframes, stream);
}

extern "C" int cm_decode_ex(cm_modem *m, const cm_window *win, const uint8_t *comp_u8, const void *comp_float,
                            uint8_t *rgb_u8, void *rgb_float, int64_t first_frame, int32_t nframes, void *stream) {
    if (!m) return fail(CM_ERR_INVALID, "null handle%s");
    return m->precision == CM_FP32
               ? run_ex<float>(m, false, win, comp_u8, comp_float, rgb_u8, rgb_float, first_frame, nframes, stream)
               : run_ex<double>(m, false, win, comp_u8, comp_float, rgb_u8, rgb_float, first_frame, nframes, stream);
}

extern "C" int cm_encode_frames(cm_modem *m, const uint8_t *rgb, uint8_t *comp, int64_t first_frame,
                                int32_t nframes, void *stream) {
    return cm_encode_ex(m, nullptr, rgb, nullptr, comp, nullptr, first_frame, nframes, stream);
}

extern "C" int cm_decode_frames(cm_modem *m, const uint8_t *comp, uint8_t *rgb, int64_t first_frame,
                                int32_t nframes, void *stream) {
    return cm_decode_ex(m, nullptr, comp, nullptr, rgb, nullptr, first_frame, nframes, stream);
}

static int ensure(void **buf, size_t *cap, size_t need) {
    if (*cap >= need) return CM_OK;
    cudaFree(*buf);
    *buf = nullptr;
    *cap = 0;
    CUDA_TRY(cudaMalloc(buf, need));
    *cap = need;
    return CM_OK;
}

// Host-buffer path shared by encode, decode and encode->decode: chunked, triple-buffered over three streams.  With pinned
// host memory the H2D copy of the next chunk, the kernels of the current one and the D2H copy of the previous one run
// concurrently (two copy engines + SMs); with pageable memory it is still correct, just serialised by the driver.
// what: 0 encode (in = RGB, out = composite), 1 decode (in = composite, out = RGB), 2 encode -> decode with the composite
// staying in device memory (in = RGB, out = RGB, mid = composite copy-out or null).
// f: picture format of the RGB side (NULL = rgb24).  For yuv420p only the 4:2:0 frames cross the link: the conversion to
// RGB runs on the kernel stream before the encoder and the one back after the decoder, through one device RGB buffer per
// staging slot; in_frame / out_frame are the link-side frame sizes.
static int run_host(cm_modem *m, int what, const uint8_t *in, uint8_t *out, uint8_t *mid, size_t in_frame, size_t out_frame,
                    size_t mid_frame, int64_t first_frame, int32_t nframes, const cm_pixfmt *f) {
    if (!m || !in || !out) return fail(CM_ERR_INVALID, "null argument%s");
    if (nframes < 0) return fail(CM_ERR_INVALID, "bad frame count%s");
    if (nframes == 0) return CM_OK;
    CUDA_TRY(cudaSetDevice(m->device));
    const bool yuv = f && f->format == CM_PIX_YUV420P;
    const int W = m->desc.width, H = m->desc.height, Wo = m->desc.out_width;
    int chunk = m->tune.host_chunk;
    if (chunk > nframes) chunk = nframes;
    for (int s = 0; s < cm_modem::kHostStreams; ++s)
        if (!m->hs[s]) CUDA_TRY(cudaStreamCreateWithFlags(&m->hs[s], cudaStreamNonBlocking));
    const bool roles = m->tune.host_roles < 0 ? what == 2 : m->tune.host_roles != 0;
    const int nbuf = roles ? cm_modem::kHostBufs : cm_modem::kHostStreams;
    for (int b = 0; b < nbuf; ++b) {
        int rc = ensure(&m->d_in[b], &m->in_cap[b], (size_t)chunk * in_frame);
        if (!rc) rc = ensure(&m->d_out[b], &m->out_cap[b], (size_t)chunk * out_frame);
        if (!rc && what == 2) rc = ensure(&m->d_mid[b], &m->mid_cap[b], (size_t)chunk * mid_frame);
        if (!rc && yuv) rc = ensure(&m->d_rgb[b], &m->rgb_cap[b], (size_t)chunk * H * (W > Wo ? W : Wo) * 3);
        if (rc) return rc;
        if (!m->ev_in[b]) {
            CUDA_TRY(cudaEventCreateWithFlags(&m->ev_in[b], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&m->ev_k[b], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&m->ev_mid[b], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&m->ev_out[b], cudaEventDisableTiming));
        }
    }
    // RGB frames the encoder reads / the decoder writes: the staging buffers themselves for rgb24, d_rgb[b] for yuv420p
    auto to_rgb = [&](const uint8_t *din, uint8_t *drgb, int n, cudaStream_t st, const uint8_t **pin) -> int {
        *pin = din;
        if (!yuv || what == 1) return CM_OK;
        *pin = drgb;
        return cm_yuv420p_to_rgb24(f, din, drgb, W, H, n, st);
    };
    auto from_rgb = [&](const uint8_t *drgb, uint8_t *dout, int n, cudaStream_t st) -> int {
        return yuv && what != 0 ? cm_rgb24_to_yuv420p(f, drgb, dout, Wo, H, n, st) : (int)CM_OK;
    };
    if (roles) {
        // One stream per role: every host->device copy on hs[0], every kernel on hs[1], every device->host copy on hs[2],
        // chained per staging buffer by events.  (With one stream per chunk the copy-in of chunk i + 3 queued behind the
        // copy-out of chunk i on the same stream, and the inbound engine idled whenever the outbound one was the busier.)
        cudaStream_t s_in = m->hs[0], s_k = m->hs[1], s_out = m->hs[2];
        int rc = CM_OK;
        cudaError_t ce = cudaSuccess;
        for (int f0 = 0, i = 0; f0 < nframes && rc == CM_OK && ce == cudaSuccess; f0 += chunk, ++i) {
            const int b = i % nbuf;
            const int n = nframes - f0 < chunk ? nframes - f0 : chunk;
            const uint8_t *din = (const uint8_t *)m->d_in[b], *pin = din;
            uint8_t *dout = (uint8_t *)m->d_out[b], *dmid = (uint8_t *)m->d_mid[b], *drgb = (uint8_t *)m->d_rgb[b];
            uint8_t *pout = yuv ? drgb : dout;
            if (i >= nbuf) ce = cudaStreamWaitEvent(s_in, m->ev_k[b], 0);             // the kernels of chunk i - nbuf have read d_in[b]
            if (ce == cudaSuccess)
                ce = cudaMemcpyAsync(m->d_in[b], in + (size_t)f0 * in_frame, (size_t)n * in_frame, cudaMemcpyHostToDevice, s_in);
            if (ce == cudaSuccess) ce = cudaEventRecord(m->ev_in[b], s_in);
            if (ce == cudaSuccess) ce = cudaStreamWaitEvent(s_k, m->ev_in[b], 0);
            if (ce == cudaSuccess && i >= nbuf) ce = cudaStreamWaitEvent(s_k, m->ev_out[b], 0);   // d_out[b] / d_mid[b] copied out
            if (ce != cudaSuccess) break;
            m->aux_slot = 1;                                                          // one kernel stream: one scratch
            rc = to_rgb(din, drgb, n, s_k, &pin);
            if (rc == CM_OK && what == 0) rc = cm_encode_frames(m, pin, dout, first_frame + f0, n, s_k);
            else if (rc == CM_OK && what == 1) rc = cm_decode_frames(m, din, pout, first_frame + f0, n, s_k);
            else if (rc == CM_OK) {
                rc = cm_encode_frames(m, pin, dmid, first_frame + f0, n, s_k);
                if (rc == CM_OK && mid) {
                    ce = cudaEventRecord(m->ev_mid[b], s_k);
                    if (ce == cudaSuccess) ce = cudaStreamWaitEvent(s_out, m->ev_mid[b], 0);
                    if (ce == cudaSuccess)
                        ce = cudaMemcpyAsync(mid + (size_t)f0 * mid_frame, dmid, (size_t)n * mid_frame, cudaMemcpyDeviceToHost, s_out);
                }
                if (rc == CM_OK && ce == cudaSuccess) rc = cm_decode_frames(m, dmid, pout, first_frame + f0, n, s_k);
            }
            if (rc == CM_OK && ce == cudaSuccess) rc = from_rgb(drgb, dout, n, s_k);
            m->aux_slot = 0;
            if (rc != CM_OK || ce != cudaSuccess) break;
            ce = cudaEventRecord(m->ev_k[b], s_k);
            if (ce == cudaSuccess) ce = cudaStreamWaitEvent(s_out, m->ev_k[b], 0);
            if (ce == cudaSuccess)
                ce = cudaMemcpyAsync(out + (size_t)f0 * out_frame, dout, (size_t)n * out_frame, cudaMemcpyDeviceToHost, s_out);
            if (ce == cudaSuccess) ce = cudaEventRecord(m->ev_out[b], s_out);
        }
        // also on failure: no copy into the caller's memory may still be in flight when this returns
        for (int s = 0; s < cm_modem::kHostStreams; ++s) {
            const cudaError_t e2 = cudaStreamSynchronize(m->hs[s]);
            if (ce == cudaSuccess) ce = e2;
        }
        if (rc != CM_OK) return rc;
        if (ce != cudaSuccess) return fail(CM_ERR_CUDA, "host path: %s", cudaGetErrorString(ce));
        return CM_OK;
    }
    int rc = CM_OK;
    cudaError_t ce = cudaSuccess;
    for (int f0 = 0, i = 0; f0 < nframes && rc == CM_OK && ce == cudaSuccess; f0 += chunk, ++i) {
        const int s = i % cm_modem::kHostStreams;
        const int n = nframes - f0 < chunk ? nframes - f0 : chunk;
        cudaStream_t st = m->hs[s];
        ce = cudaMemcpyAsync(m->d_in[s], in + (size_t)f0 * in_frame, (size_t)n * in_frame, cudaMemcpyHostToDevice, st);
        if (ce != cudaSuccess) break;
        m->aux_slot = 1 + s;
        const uint8_t *din = (const uint8_t *)m->d_in[s], *pin = din;
        uint8_t *dout = (uint8_t *)m->d_out[s], *dmid = (uint8_t *)m->d_mid[s], *drgb = (uint8_t *)m->d_rgb[s];
        uint8_t *pout = yuv ? drgb : dout;
        rc = to_rgb(din, drgb, n, st, &pin);
        if (rc == CM_OK && what == 0) rc = cm_encode_frames(m, pin, dout, first_frame + f0, n, st);
        else if (rc == CM_OK && what == 1) rc = cm_decode_frames(m, din, pout, first_frame + f0, n, st);
        else if (rc == CM_OK) {
            rc = cm_encode_frames(m, pin, dmid, first_frame + f0, n, st);
            if (rc == CM_OK && mid)
                ce = cudaMemcpyAsync(mid + (size_t)f0 * mid_frame, dmid, (size_t)n * mid_frame, cudaMemcpyDeviceToHost, st);
            if (rc == CM_OK) rc = cm_decode_frames(m, dmid, pout, first_frame + f0, n, st);
        }
        if (rc == CM_OK && ce == cudaSuccess) rc = from_rgb(drgb, dout, n, st);
        m->aux_slot = 0;
        if (rc == CM_OK && ce == cudaSuccess)
            ce = cudaMemcpyAsync(out + (size_t)f0 * out_frame, dout, (size_t)n * out_frame, cudaMemcpyDeviceToHost, st);
    }
    // also on failure: no copy into the caller's memory may still be in flight when this returns
    for (int s = 0; s < cm_modem::kHostStreams; ++s) {
        const cudaError_t e2 = cudaStreamSynchronize(m->hs[s]);
        if (ce == cudaSuccess) ce = e2;
    }
    if (rc != CM_OK) return rc;
    if (ce != cudaSuccess) return fail(CM_ERR_CUDA, "host path: %s", cudaGetErrorString(ce));
    return CM_OK;
}

// Bytes of one picture-side frame w wide in format f (NULL = rgb24); 0 for a format that does not exist.
static size_t pic_frame(const cm_pixfmt *f, int w, int h) {
    if (!f || f->format == CM_PIX_RGB24) return (size_t)h * w * 3;
    if (f->format != CM_PIX_YUV420P || f->reserved || (f->matrix != CM_YUV_BT601 && f->matrix != CM_YUV_BT709) ||
        (f->range != CM_YUV_LIMITED && f->range != CM_YUV_FULL))
        return 0;
    return (size_t)h * w + (size_t)w * ((h + 1) / 2);        // Y + U + V: W H + 2 (W/2) ceil(H/2)
}

extern "C" int cm_encode_frames_host_fmt(cm_modem *m, const uint8_t *pic, uint8_t *comp, int64_t first_frame,
                                         int32_t nframes, const cm_pixfmt *f) {
    if (!m) return fail(CM_ERR_INVALID, "null handle%s");
    const size_t in_frame = pic_frame(f, m->desc.width, m->desc.height);
    if (!in_frame) return fail(CM_ERR_INVALID, "bad cm_pixfmt%s");
    return run_host(m, 0, pic, comp, nullptr, in_frame, (size_t)m->desc.height * m->desc.comp_width, 0, first_frame, nframes,
                    f);
}

extern "C" int cm_decode_frames_host_fmt(cm_modem *m, const uint8_t *comp, uint8_t *pic, int64_t first_frame,
                                         int32_t nframes, const cm_pixfmt *f) {
    if (!m) return fail(CM_ERR_INVALID, "null handle%s");
    const size_t out_frame = pic_frame(f, m->desc.out_width, m->desc.height);
    if (!out_frame) return fail(CM_ERR_INVALID, "bad cm_pixfmt%s");
    return run_host(m, 1, comp, pic, nullptr, (size_t)m->desc.height * m->desc.comp_width, out_frame, 0, first_frame, nframes,
                    f);
}

extern "C" int cm_transcode_frames_host_fmt(cm_modem *m, const uint8_t *pic_in, uint8_t *comp_out, uint8_t *pic_out,
                                            int64_t first_frame, int32_t nframes, const cm_pixfmt *f) {
    if (!m) return fail(CM_ERR_INVALID, "null handle%s");
    const size_t in_frame = pic_frame(f, m->desc.width, m->desc.height), out_frame = pic_frame(f, m->desc.out_width, m->desc.height);
    if (!in_frame) return fail(CM_ERR_INVALID, "bad cm_pixfmt%s");
    return run_host(m, 2, pic_in, pic_out, comp_out, in_frame, out_frame, (size_t)m->desc.height * m->desc.comp_width,
                    first_frame, nframes, f);
}

extern "C" int cm_encode_frames_host(cm_modem *m, const uint8_t *rgb, uint8_t *comp, int64_t first_frame,
                                     int32_t nframes) {
    return cm_encode_frames_host_fmt(m, rgb, comp, first_frame, nframes, nullptr);
}

extern "C" int cm_decode_frames_host(cm_modem *m, const uint8_t *comp, uint8_t *rgb, int64_t first_frame,
                                     int32_t nframes) {
    return cm_decode_frames_host_fmt(m, comp, rgb, first_frame, nframes, nullptr);
}

extern "C" int cm_transcode_frames_host(cm_modem *m, const uint8_t *rgb_in, uint8_t *comp_out, uint8_t *rgb_out,
                                        int64_t first_frame, int32_t nframes) {
    return cm_transcode_frames_host_fmt(m, rgb_in, comp_out, rgb_out, first_frame, nframes, nullptr);
}
