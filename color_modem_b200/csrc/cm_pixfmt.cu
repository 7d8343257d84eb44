// Picture formats of the frame-batch paths: planar YUV 4:2:0 (I420, `yuv420p`) <-> packed RGB24, in Q16 integer arithmetic
// (the definition, and its numpy restatement, in oracle/yuv.py; INTEGRATION.md "Picture formats").
//
// Layout of one yuv420p frame: Y [H][W], then U [ceil(H/2)][W/2], then V [ceil(H/2)][W/2].  W is a multiple of 4, so a luma
// row and a group of four RGB pixels (12 bytes) are 4-byte aligned; W/2 may be 2 mod 4, so a chroma row is only 2-byte
// aligned and every chroma access here is 16-bit.  One thread owns four pixels of a row pair: two 32-bit luma words, one
// 16-bit word each of U and V (the two chroma samples of that 4x2 block), three 32-bit RGB words per row.
#include "cm_host.h"

struct YuvCoef {
    int oY;
    int YR, YG, YB, UR, UG, UB, VR, VG, VB;      // RGB -> YUV
    int Y, RV, GU, GV, BU;                         // YUV -> RGB
};

static int round_half_away(double x) { return (int)(x < 0 ? -floor(-x + 0.5) : floor(x + 0.5)); }

// The coefficient rule of oracle/yuv.py, term for term in the same float64 expressions.
static int pix_coef(const cm_pixfmt *f, YuvCoef &c) {
    if (!f) return cm_fail(CM_ERR_INVALID, "null cm_pixfmt%s");
    if (f->format != CM_PIX_YUV420P) return cm_fail(CM_ERR_INVALID, "cm_pixfmt.format must be CM_PIX_YUV420P here%s");
    if (f->matrix != CM_YUV_BT601 && f->matrix != CM_YUV_BT709) return cm_fail(CM_ERR_INVALID, "bad cm_pixfmt.matrix%s");
    if (f->range != CM_YUV_LIMITED && f->range != CM_YUV_FULL) return cm_fail(CM_ERR_INVALID, "bad cm_pixfmt.range%s");
    if (f->reserved) return cm_fail(CM_ERR_INVALID, "cm_pixfmt.reserved must be 0%s");
    const double kr = f->matrix == CM_YUV_BT601 ? 0.299 : 0.2126, kb = f->matrix == CM_YUV_BT601 ? 0.114 : 0.0722;
    const double kg = 1.0 - kr - kb;
    const bool limited = f->range == CM_YUV_LIMITED;
    const double sy = limited ? 219.0 / 255.0 : 1.0, sc = limited ? 224.0 / 255.0 : 1.0, q = 65536.0;
    c.oY = limited ? 16 : 0;
    c.YR = round_half_away(q * sy * kr);
    c.YB = round_half_away(q * sy * kb);
    c.YG = round_half_away(q * sy) - c.YR - c.YB;
    c.UR = round_half_away(q * sc * -kr / (2.0 * (1.0 - kb)));
    c.UB = round_half_away(q * sc * 0.5);
    c.UG = -(c.UR + c.UB);
    c.VR = round_half_away(q * sc * 0.5);
    c.VB = round_half_away(q * sc * -kb / (2.0 * (1.0 - kr)));
    c.VG = -(c.VR + c.VB);
    const double iy = limited ? 255.0 / 219.0 : 1.0, ic = limited ? 255.0 / 224.0 : 1.0;
    c.Y = round_half_away(q * iy);
    c.RV = round_half_away(q * ic * 2.0 * (1.0 - kr));
    c.GU = round_half_away(q * ic * -2.0 * kb * (1.0 - kb) / kg);
    c.GV = round_half_away(q * ic * -2.0 * kr * (1.0 - kr) / kg);
    c.BU = round_half_away(q * ic * 2.0 * (1.0 - kb));
    return CM_OK;
}

__device__ __forceinline__ uint32_t clip8(int v) { return (uint32_t)min(max(v, 0), 255); }

// Pixel k of a 12-byte RGB group lives in bytes 3k .. 3k + 2 of the three little-endian words.
__device__ __forceinline__ void pack_rgb(const uint32_t r[4], const uint32_t g[4], const uint32_t b[4], uint32_t w[3]) {
    w[0] = r[0] | g[0] << 8 | b[0] << 16 | r[1] << 24;
    w[1] = g[1] | b[1] << 8 | r[2] << 16 | g[2] << 24;
    w[2] = b[2] | r[3] << 8 | g[3] << 16 | b[3] << 24;
}

__device__ __forceinline__ void unpack_rgb(const uint32_t w[3], int r[4], int g[4], int b[4]) {
    r[0] = w[0] & 255; g[0] = w[0] >> 8 & 255; b[0] = w[0] >> 16 & 255; r[1] = w[0] >> 24;
    g[1] = w[1] & 255; b[1] = w[1] >> 8 & 255; r[2] = w[1] >> 16 & 255; g[2] = w[1] >> 24;
    b[2] = w[2] & 255; r[3] = w[2] >> 8 & 255; g[3] = w[2] >> 16 & 255; b[3] = w[2] >> 24;
}

// grid: x = ceil(W/4 * ceil(H/2) / blockDim.x), z = frame
__global__ void __launch_bounds__(256)
k_yuv420p_to_rgb24(const YuvCoef c, const uint8_t *__restrict__ yuv, uint8_t *__restrict__ rgb, int W, int H) {
    const int gw = W >> 2, hc = (H + 1) >> 1;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= gw * hc) return;
    const int py = t / gw, gx = t - py * gw;
    const size_t plane = (size_t)W * H, cplane = (size_t)(W >> 1) * hc;
    const uint8_t *src = yuv + (size_t)blockIdx.z * (plane + 2 * cplane);
    uint8_t *dst = rgb + (size_t)blockIdx.z * plane * 3;
    const size_t co = (size_t)py * (W >> 1) + 2 * gx;
    const uint32_t u2 = *reinterpret_cast<const uint16_t *>(src + plane + co);
    const uint32_t v2 = *reinterpret_cast<const uint16_t *>(src + plane + cplane + co);
    int cr[2], cg[2], cb[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const int u = (int)(u2 >> 8 * k & 255) - 128, v = (int)(v2 >> 8 * k & 255) - 128;
        cr[k] = c.RV * v + 32768;
        cg[k] = c.GU * u + c.GV * v + 32768;
        cb[k] = c.BU * u + 32768;
    }
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
        const int y = 2 * py + dy;
        if (y >= H) break;
        const uint32_t l4 = *reinterpret_cast<const uint32_t *>(src + (size_t)y * W + 4 * gx);
        uint32_t r[4], g[4], b[4], w[3];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int ly = c.Y * ((int)(l4 >> 8 * k & 255) - c.oY);
            r[k] = clip8((ly + cr[k >> 1]) >> 16);
            g[k] = clip8((ly + cg[k >> 1]) >> 16);
            b[k] = clip8((ly + cb[k >> 1]) >> 16);
        }
        pack_rgb(r, g, b, w);
        uint32_t *o = reinterpret_cast<uint32_t *>(dst + ((size_t)y * W + 4 * gx) * 3);
        o[0] = w[0];
        o[1] = w[1];
        o[2] = w[2];
    }
}

__global__ void __launch_bounds__(256)
k_rgb24_to_yuv420p(const YuvCoef c, const uint8_t *__restrict__ rgb, uint8_t *__restrict__ yuv, int W, int H) {
    const int gw = W >> 2, hc = (H + 1) >> 1;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= gw * hc) return;
    const int py = t / gw, gx = t - py * gw;
    const size_t plane = (size_t)W * H, cplane = (size_t)(W >> 1) * hc;
    const uint8_t *src = rgb + (size_t)blockIdx.z * plane * 3;
    uint8_t *dst = yuv + (size_t)blockIdx.z * (plane + 2 * cplane);
    int su[2] = {0, 0}, sv[2] = {0, 0};
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
        const int y = 2 * py + dy < H ? 2 * py + dy : H - 1;        // odd height: the last row stands in for the missing one
        const uint32_t *in = reinterpret_cast<const uint32_t *>(src + ((size_t)y * W + 4 * gx) * 3);
        const uint32_t w[3] = {in[0], in[1], in[2]};
        int r[4], g[4], b[4];
        unpack_rgb(w, r, g, b);
        uint32_t l4 = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            l4 |= clip8((c.YR * r[k] + c.YG * g[k] + c.YB * b[k] + c.oY * 65536 + 32768) >> 16) << 8 * k;
            su[k >> 1] += c.UR * r[k] + c.UG * g[k] + c.UB * b[k];
            sv[k >> 1] += c.VR * r[k] + c.VG * g[k] + c.VB * b[k];
        }
        if (2 * py + dy < H) *reinterpret_cast<uint32_t *>(dst + (size_t)y * W + 4 * gx) = l4;
    }
    const size_t co = (size_t)py * (W >> 1) + 2 * gx;
    const int bias = 128 * (1 << 18) + (1 << 17);
    *reinterpret_cast<uint16_t *>(dst + plane + co) =
        (uint16_t)(clip8((su[0] + bias) >> 18) | clip8((su[1] + bias) >> 18) << 8);
    *reinterpret_cast<uint16_t *>(dst + plane + cplane + co) =
        (uint16_t)(clip8((sv[0] + bias) >> 18) | clip8((sv[1] + bias) >> 18) << 8);
}

static int pix_convert(bool to_rgb, const cm_pixfmt *f, const uint8_t *src, uint8_t *dst, int32_t width, int32_t height,
                       int32_t nframes, void *stream) {
    YuvCoef c;
    int rc = pix_coef(f, c);
    if (rc) return rc;
    if (width <= 0 || height <= 0 || (width & 3)) return cm_fail(CM_ERR_INVALID, "width must be a positive multiple of 4%s");
    if (nframes < 0) return cm_fail(CM_ERR_INVALID, "bad frame count%s");
    if (nframes == 0) return CM_OK;
    if (!src || !dst) return cm_fail(CM_ERR_INVALID, "null buffer%s");
    const long long threads = (long long)(width >> 2) * ((height + 1) >> 1);
    if (threads > 0x7fffffffLL) return cm_fail(CM_ERR_INVALID, "frame too large%s");
    const size_t in_frame = to_rgb ? (size_t)width * height + (size_t)width * ((height + 1) >> 1) : (size_t)width * height * 3;
    const size_t out_frame = to_rgb ? (size_t)width * height * 3 : (size_t)width * height + (size_t)width * ((height + 1) >> 1);
    const unsigned bx = (unsigned)((threads + 255) / 256);
    for (int32_t base = 0; base < nframes; base += 65535) {         // gridDim.z carries the frame index
        const unsigned nz = (unsigned)(nframes - base < 65535 ? nframes - base : 65535);
        const uint8_t *s = src + (size_t)base * in_frame;
        uint8_t *d = dst + (size_t)base * out_frame;
        if (to_rgb) k_yuv420p_to_rgb24<<<dim3(bx, 1, nz), 256, 0, (cudaStream_t)stream>>>(c, s, d, width, height);
        else k_rgb24_to_yuv420p<<<dim3(bx, 1, nz), 256, 0, (cudaStream_t)stream>>>(c, s, d, width, height);
        cm_count_launch();
        CUDA_TRY(cudaGetLastError());
    }
    return CM_OK;
}

extern "C" int cm_yuv420p_to_rgb24(const cm_pixfmt *f, const uint8_t *yuv, uint8_t *rgb, int32_t width, int32_t height,
                                   int32_t nframes, void *stream) {
    return pix_convert(true, f, yuv, rgb, width, height, nframes, stream);
}

extern "C" int cm_rgb24_to_yuv420p(const cm_pixfmt *f, const uint8_t *rgb, uint8_t *yuv, int32_t width, int32_t height,
                                   int32_t nframes, void *stream) {
    return pix_convert(false, f, rgb, yuv, width, height, nframes, stream);
}
