/* jfif_oracle.c — TEST INFRASTRUCTURE: a scalar restatement of libjpeg-turbo's default RGB output stage (the libjpeg
 * colour convention, ROCJPEG_B200_COLOR_LIBJPEG): chroma upsampling as jdsample.c's jinit_upsampler picks it and
 * jdcolor.c's JFIF integer YCbCr -> RGB conversion, applied to the oracle's component planes (full size, or the reduced-size
 * planes of tests/scaled_oracle.c). Compiled together with the unchanged oracle source (oracle/jpeg_oracle.c, included
 * below) into its own library: it uses the oracle's OrcInfo and ROI rule, and assembles RGB / RGB_PLANAR with orc_convert's
 * crop and pitch rules (the crop is a window of the uncropped result).
 *
 * Upsampling of a component with expansion hr x vr (hmax / h, vmax / v), downsampled size cw = ceil(W / hr),
 * ch = ceil(H / vr) (W x H = the output size), neighbour indices clamped into [0, cw) x [0, ch):
 *   2x1 h2v1_fancy: (3 c[i] + c[i-1] + 1) >> 2 (even column), (3 c[i] + c[i+1] + 2) >> 2 (odd column);
 *   1x2 h1v2_fancy: (3 c[k] + c[k-1] + 1) >> 2 (upper row), (3 c[k] + c[k+1] + 2) >> 2 (lower row);
 *   2x2 h2v2_fancy: colsum = 3 c[k] + c[k-1] (upper) or 3 c[k] + c[k+1] (lower); (3 colsum[i] + colsum[i-1] + 8) >> 4
 *       (even column), (3 colsum[i] + colsum[i+1] + 7) >> 4 (odd column);
 *   everything else replicates: 1x1, 4x1 (int_upsample), a 1x1 transform (do_fancy needs min_DCT_scaled_size > 1), and
 *   2x1 / 2x2 with cw <= 2. */
#include "jpeg_oracle.c"

static inline uint8_t jfif_clamp(int v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

/* Upsampled chroma sample (X, Y) of plane c (rows `pitch` apart). fancy: the transform is larger than 1x1. */
static int jfif_chroma(const uint8_t *pl, int pitch, int hr, int vr, int cw, int ch, int fancy, int X, int Y) {
#define AT(i, k) ((int)pl[(size_t)(k) * pitch + (i)])
#define CL(v, n) ((v) < 0 ? 0 : ((v) >= (n) ? (n) - 1 : (v)))
    if (fancy && hr == 2 && vr == 1 && cw > 2) {
        int i = X >> 1, k = Y;
        return (X & 1) ? (3 * AT(i, k) + AT(CL(i + 1, cw), k) + 2) >> 2 : (3 * AT(i, k) + AT(CL(i - 1, cw), k) + 1) >> 2;
    }
    if (fancy && hr == 1 && vr == 2) {
        int i = X, k = Y >> 1;
        return (Y & 1) ? (3 * AT(i, k) + AT(i, CL(k + 1, ch)) + 2) >> 2 : (3 * AT(i, k) + AT(i, CL(k - 1, ch)) + 1) >> 2;
    }
    if (fancy && hr == 2 && vr == 2 && cw > 2) {
        int i = X >> 1, k = Y >> 1, kn = (Y & 1) ? CL(k + 1, ch) : CL(k - 1, ch);
        int in = (X & 1) ? CL(i + 1, cw) : CL(i - 1, cw);
        int cs = 3 * AT(i, k) + AT(i, kn), csn = 3 * AT(in, k) + AT(in, kn);
        return (X & 1) ? (3 * cs + csn + 7) >> 4 : (3 * cs + csn + 8) >> 4;
    }
    return AT(X / hr, Y / vr);
#undef AT
#undef CL
}

/* planes: orc_idct_planes' layout (component c is blocks_h[c]*8 rows of blocks_w[c]*8 samples; at scale 1/d its top-left
 * (8/d)-per-block corner holds the reduced-size plane). o: the info at the output size (W x H at scale 1/d).
 * fmt: FMT_RGB or FMT_RGB_PLANAR; crop, dst, dst_pitch: as orc_convert. */
int jfif_convert(const OrcInfo *o, const uint8_t *planes, int d, int fmt, const int16_t crop[4], uint8_t *dst[4],
                 const uint32_t dst_pitch[4]) {
    if (fmt != FMT_RGB && fmt != FMT_RGB_PLANAR) return ORC_INVALID;
    const uint8_t *pl[3] = {NULL, NULL, NULL};
    int pitch[3] = {0, 0, 0};
    size_t cb = 0;
    for (int c = 0; c < o->ncomp; c++) {
        pl[c] = planes + cb;
        pitch[c] = o->blocks_w[c] * 8;
        cb += (size_t)o->blocks_w[c] * o->blocks_h[c] * 64;
    }
    int x0, y0, W, H;
    if (orc_roi(o, crop, &x0, &y0, &W, &H) < 0) return ORC_INVALID;
    if (fmt == FMT_RGB && (!dst[0] || !dst_pitch[0])) return ORC_OK;
    if (fmt == FMT_RGB_PLANAR && (!dst[0] || !dst[1] || !dst[2] || !dst_pitch[0])) return ORC_OK;
    const int gray = o->ncomp == 1, fancy = d < 8;
    int hr = 1, vr = 1, cw = 0, ch = 0;
    if (!gray) {
        hr = o->hmax / o->hs[1];
        vr = o->vmax / o->vs[1];
        cw = (o->width + hr - 1) / hr;
        ch = (o->height + vr - 1) / vr;
    }
    for (int y = 0; y < H; y++)
        for (int x = 0; x < W; x++) {
            const int X = x0 + x, Y = y0 + y;
            const int yy = pl[0][(size_t)Y * pitch[0] + X];
            uint8_t r, g, b;
            if (gray) {
                r = g = b = (uint8_t)yy;
            } else {
                const int u = jfif_chroma(pl[1], pitch[1], hr, vr, cw, ch, fancy, X, Y) - 128;
                const int v = jfif_chroma(pl[2], pitch[2], hr, vr, cw, ch, fancy, X, Y) - 128;
                r = jfif_clamp(yy + ((91881 * v + 32768) >> 16));
                g = jfif_clamp(yy + ((-22554 * u - 46802 * v + 32768) >> 16));
                b = jfif_clamp(yy + ((116130 * u + 32768) >> 16));
            }
            if (fmt == FMT_RGB) {
                uint8_t *p = dst[0] + (size_t)y * dst_pitch[0] + 3 * x;
                p[0] = r; p[1] = g; p[2] = b;
            } else { /* all three planes use pitch[0] */
                dst[0][(size_t)y * dst_pitch[0] + x] = r;
                dst[1][(size_t)y * dst_pitch[0] + x] = g;
                dst[2][(size_t)y * dst_pitch[0] + x] = b;
            }
        }
    return ORC_OK;
}
