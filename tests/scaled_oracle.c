/* scaled_oracle.c — TEST INFRASTRUCTURE: the oracle's restatement of the reduced-size IDCTs used by decodes at 1/2,
 * 1/4 and 1/8 scale. It is compiled together with the unchanged oracle source (oracle/jpeg_oracle.c, included
 * below) into its own library, so it works on the oracle's OrcInfo, zig-zag table and islow block as they are.
 *
 * libjpeg's jidctred.c (jpeg_idct_4x4, jpeg_idct_2x2, jpeg_idct_1x1), which libjpeg-turbo uses for scale_num = 1,
 * scale_denom = 2, 4, 8. CONST_BITS 13, PASS1_BITS 2. Their zero-AC shortcuts are arithmetically identical to the
 * general path and are not taken. Like the oracle's islow restatement: 32-bit intermediates, and the output saturates
 * to 0..255 (libjpeg indexes a range-limit table with the value masked to 10 bits, which agrees with saturation for
 * every value a valid stream produces). */
#include "jpeg_oracle.c"

#define FIX_0_211164243 1730
#define FIX_0_509795579 4176
#define FIX_0_601344887 4926
#define FIX_0_720959822 5906
#define FIX_0_850430095 6967
#define FIX_1_061594337 8697
#define FIX_1_272758580 10426
#define FIX_1_451774981 11893
#define FIX_2_172734803 17799
#define FIX_3_624509785 29692

static inline uint8_t sat_u8(int32_t v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }
#define DESCALE(x, n) (((x) + (1 << ((n) - 1))) >> (n))

/* in[0..7] = positions 0..7 of a row or column (position 4 is not read); out[0..3] */
static inline void red4_1d(const int32_t in[8], int32_t out[4], int shift) {
    int32_t tmp0 = in[0] * (1 << 14); /* << (CONST_BITS + 1) */
    int32_t tmp2 = in[2] * FIX_1_847759065 + in[6] * (-FIX_0_765366865);
    int32_t tmp10 = tmp0 + tmp2, tmp12 = tmp0 - tmp2;
    int32_t z1 = in[7], z2 = in[5], z3 = in[3], z4 = in[1];
    tmp0 = z1 * (-FIX_0_211164243) + z2 * FIX_1_451774981 + z3 * (-FIX_2_172734803) + z4 * FIX_1_061594337;
    tmp2 = z1 * (-FIX_0_509795579) + z2 * (-FIX_0_601344887) + z3 * FIX_0_899976223 + z4 * FIX_2_562915447;
    out[0] = DESCALE(tmp10 + tmp2, shift);
    out[3] = DESCALE(tmp10 - tmp2, shift);
    out[1] = DESCALE(tmp12 + tmp0, shift);
    out[2] = DESCALE(tmp12 - tmp0, shift);
}

/* in[0..7] = positions 0..7 (only 0, 1, 3, 5, 7 are read); out[0..1] */
static inline void red2_1d(const int32_t in[8], int32_t out[2], int shift) {
    int32_t tmp10 = in[0] * (1 << 15); /* << (CONST_BITS + 2) */
    int32_t tmp0 = in[7] * (-FIX_0_720959822) + in[5] * FIX_0_850430095 + in[3] * (-FIX_1_272758580) + in[1] * FIX_3_624509785;
    out[0] = DESCALE(tmp10 + tmp0, shift);
    out[1] = DESCALE(tmp10 - tmp0, shift);
}

/* One block at scale 1/d (d = 1, 2, 4, 8): an (8/d) x (8/d) square of samples at `out`, rows `pitch` apart. */
void orc_idct_scaled_block(const int16_t *coef, const uint16_t *q_nat, int d, uint8_t *out, int pitch) {
    if (d == 1) {
        orc_idct_islow_block(coef, q_nat, out, pitch);
        return;
    }
    if (d == 8) { /* jpeg_idct_1x1 */
        int32_t dc = (int32_t)coef[0] * (int32_t)q_nat[0];
        out[0] = sat_u8(DESCALE(dc, 3) + 128);
        return;
    }
    const int S = 8 / d;
    int32_t ws[8 * 8], col[8], res[4];
    for (int c = 0; c < 8; c++) { /* pass 1: columns, descaled by CONST_BITS - PASS1_BITS + log2(d) */
        for (int r = 0; r < 8; r++) col[r] = (int32_t)coef[r * 8 + c] * (int32_t)q_nat[r * 8 + c];
        if (S == 4) red4_1d(col, res, 13 - 2 + 1);
        else red2_1d(col, res, 13 - 2 + 2);
        for (int r = 0; r < S; r++) ws[r * 8 + c] = res[r];
    }
    for (int r = 0; r < S; r++) { /* pass 2: rows, descaled by CONST_BITS + PASS1_BITS + 3 + log2(d) */
        if (S == 4) red4_1d(ws + r * 8, res, 13 + 2 + 3 + 1);
        else red2_1d(ws + r * 8, res, 13 + 2 + 3 + 2);
        for (int c = 0; c < S; c++) out[r * pitch + c] = sat_u8(res[c] + 128);
    }
}

/* orc_idct_planes at scale 1/d. planes: the layout of orc_idct_planes (component-major, each plane
 * (blocks_w*8) x (blocks_h*8) bytes, pitch blocks_w*8); the scaled plane, (blocks_w*8/d) x (blocks_h*8/d)
 * samples, occupies its top-left corner at the same pitch - so orc_convert assembles the output of a scaled
 * decode from it unchanged, given an OrcInfo whose width / height are the scaled ones. */
int orc_idct_planes_scaled(const OrcInfo *o, const int16_t *coefs, int d, uint8_t *planes) {
    if (d != 1 && d != 2 && d != 4 && d != 8) return ORC_INVALID;
    const int S = 8 / d;
    size_t cb = 0;
    for (int c = 0; c < o->ncomp; c++) {
        uint16_t qn[64];
        for (int k = 0; k < 64; k++) qn[kZigzag[k]] = o->qt16[o->tq[c]][k];
        int pitch = o->blocks_w[c] * 8;
        for (int by = 0; by < o->blocks_h[c]; by++)
            for (int bx = 0; bx < o->blocks_w[c]; bx++) {
                const int16_t *blk = coefs + cb + ((size_t)by * o->blocks_w[c] + bx) * 64;
                orc_idct_scaled_block(blk, qn, d, planes + cb + (size_t)by * S * pitch + bx * S, pitch);
            }
        cb += (size_t)o->blocks_w[c] * o->blocks_h[c] * 64;
    }
    return ORC_OK;
}
