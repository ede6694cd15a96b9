/* ljt_scaled.c — TEST INFRASTRUCTURE: libjpeg-turbo at scale 1/2, 1/4, 1/8 (scale_num = 1, scale_denom = d), to pin
 * the oracle's reduced-size IDCTs and as the CPU baseline of scaled decodes. It is compiled together with the unchanged
 * header-less harness (oracle/ljt_shim.c, included below) into its own library and uses that harness's hand-declared
 * struct offsets, adding the few that scaling needs; ljt_selfcheck() verifies those on a stream at run time. */
#include "ljt_shim.c"

#define OFF_SCALE_NUM 68
#define OFF_SCALE_DENOM 72
#define COMP_DCT_SCALED_SIZE 36

/* Raw planes at scale 1/d: libjpeg-turbo transforms every block of component c with the reduced IDCT of size
 * DCT_scaled_size (returned in dss[c]; for 4:2:0 chroma it is twice the luma size, jdmaster.c). planes: the layout of
 * ljt_read_raw (component-major, plane c (bw[c]*8) x (bh[c]*8) bytes); the scaled plane, (bw[c]*dss[c]) x
 * (bh[c]*dss[c]), occupies its top-left corner at pitch bw[c]*8. Only the wib x hib blocks' part of it is defined. */
int ljt_read_raw_scaled(const uint8_t *data, size_t len, int d, uint8_t *planes, const int32_t bw[3], const int32_t bh[3],
                        int32_t dss[3]) {
    char ci[CINFO_SIZE + 64];
    ErrCtx e;
    uint8_t **rowptr[3] = {0, 0, 0};
    setup(ci, &e);
    if (setjmp(e.jb)) {
        L.destroy(ci);
        for (int c = 0; c < 3; c++) free(rowptr[c]);
        return -1;
    }
    L.mem_src(ci, data, (unsigned long)len);
    L.read_header(ci, 1);
    I32(ci, OFF_RAW_DATA_OUT) = 1;
    I32(ci, OFF_DCT_METHOD) = 0; /* JDCT_ISLOW */
    U32(ci, OFF_SCALE_NUM) = 1;
    U32(ci, OFF_SCALE_DENOM) = (uint32_t)d;
    int ncomp = I32(ci, OFF_NUM_COMPONENTS);
    L.start(ci);
    char *comp = (char *)PTR(ci, OFF_COMP_INFO);
    int vmax = 1, vs[3] = {1, 1, 1}, min_dss = 8;
    uint8_t *pbase[3];
    size_t base = 0;
    for (int c = 0; c < ncomp && c < 3; c++) {
        vs[c] = I32(comp + c * COMP_STRIDE, COMP_V);
        dss[c] = I32(comp + c * COMP_STRIDE, COMP_DCT_SCALED_SIZE);
        if (vs[c] > vmax) vmax = vs[c];
        if (dss[c] < min_dss) min_dss = dss[c];
        pbase[c] = planes + base;
        base += (size_t)bw[c] * bh[c] * 64;
        rowptr[c] = (uint8_t **)malloc(sizeof(uint8_t *) * 8 * 4);
    }
    unsigned out_h = U32(ci, OFF_OUTPUT_HEIGHT);
    int imcu = 0;
    while (U32(ci, OFF_OUTPUT_SCANLINE) < out_h) {
        for (int c = 0; c < ncomp && c < 3; c++)
            for (int r = 0; r < vs[c] * dss[c]; r++) {
                size_t row = (size_t)imcu * vs[c] * dss[c] + r;
                rowptr[c][r] = pbase[c] + row * (size_t)bw[c] * 8;
            }
        unsigned got = L.read_raw(ci, rowptr, (unsigned)(vmax * min_dss));
        if (!got) break;
        imcu++;
    }
    L.finish(ci);
    L.destroy(ci);
    for (int c = 0; c < 3; c++) free(rowptr[c]);
    return 0;
}

/* output_width / output_height libjpeg-turbo computes for scale 1/d (jpeg_calc_output_dimensions). */
int ljt_output_size(const uint8_t *data, size_t len, int d, int32_t wh[2]) {
    char ci[CINFO_SIZE + 64];
    ErrCtx e;
    setup(ci, &e);
    if (setjmp(e.jb)) { L.destroy(ci); return -1; }
    L.mem_src(ci, data, (unsigned long)len);
    L.read_header(ci, 1);
    U32(ci, OFF_SCALE_NUM) = 1;
    U32(ci, OFF_SCALE_DENOM) = (uint32_t)d;
    L.start(ci);
    wh[0] = (int32_t)U32(ci, OFF_OUTPUT_WIDTH);
    wh[1] = (int32_t)U32(ci, OFF_OUTPUT_HEIGHT);
    L.abort_(ci);
    L.destroy(ci);
    return 0;
}

/* Checks the struct offsets the scaled decodes rely on, on one stream: scale_num / scale_denom read 1 / 1 after
 * jpeg_read_header; with 1/2 set, jpeg_start_decompress reports output_width / output_height = ceil(W/2) / ceil(H/2)
 * and a DCT_scaled_size of 4 for the first component. 0: all hold. */
int ljt_selfcheck(const uint8_t *data, size_t len) {
    char ci[CINFO_SIZE + 64];
    ErrCtx e;
    setup(ci, &e);
    if (setjmp(e.jb)) { L.destroy(ci); return -1; }
    L.mem_src(ci, data, (unsigned long)len);
    L.read_header(ci, 1);
    int rc = 0;
    if (U32(ci, OFF_SCALE_NUM) != 1 || U32(ci, OFF_SCALE_DENOM) != 1) rc = -2;
    unsigned w = U32(ci, OFF_IMAGE_WIDTH), h = U32(ci, OFF_IMAGE_HEIGHT);
    I32(ci, OFF_RAW_DATA_OUT) = 1;
    U32(ci, OFF_SCALE_DENOM) = 2;
    L.start(ci);
    if (!rc && (U32(ci, OFF_OUTPUT_WIDTH) != (w + 1) / 2 || U32(ci, OFF_OUTPUT_HEIGHT) != (h + 1) / 2)) rc = -3;
    if (!rc && I32((char *)PTR(ci, OFF_COMP_INFO), COMP_DCT_SCALED_SIZE) != 4) rc = -4;
    L.abort_(ci);
    L.destroy(ci);
    return rc;
}

/* libjpeg-turbo's default decode at scale 1/d. mode 0: ceil(W/d) x ceil(H/d) RGB pixels into out (pitch bytes/row);
 * mode 2: raw planes (ljt_read_raw_scaled into a scratch of sum(bw*bh*64)). */
static int decode_one_scaled(const uint8_t *data, size_t len, uint8_t *out, size_t pitch, int mode, int d) {
    char ci[CINFO_SIZE + 64];
    ErrCtx e;
    setup(ci, &e);
    if (setjmp(e.jb)) { L.destroy(ci); return -1; }
    L.mem_src(ci, data, (unsigned long)len);
    L.read_header(ci, 1);
    if (mode == 2) {
        LjtInfo inf;
        fill_info(ci, &inf);
        L.destroy(ci);
        int32_t bw[3] = {0, 0, 0}, bh[3] = {0, 0, 0}, dss[3];
        int hmax = 1, vmax = 1;
        for (int c = 0; c < inf.ncomp && c < 3; c++) {
            if (inf.hs[c] > hmax) hmax = inf.hs[c];
            if (inf.vs[c] > vmax) vmax = inf.vs[c];
        }
        int mx = (inf.width + 8 * hmax - 1) / (8 * hmax), my = (inf.height + 8 * vmax - 1) / (8 * vmax);
        for (int c = 0; c < inf.ncomp && c < 3; c++) {
            bw[c] = (inf.ncomp == 1) ? (inf.width + 7) / 8 : mx * inf.hs[c];
            bh[c] = (inf.ncomp == 1) ? (inf.height + 7) / 8 : my * inf.vs[c];
        }
        return ljt_read_raw_scaled(data, len, d, out, bw, bh, dss);
    }
    I32(ci, OFF_OUT_COLOR_SPACE) = 2; /* JCS_RGB */
    U32(ci, OFF_SCALE_NUM) = 1;
    U32(ci, OFF_SCALE_DENOM) = (uint32_t)d;
    L.start(ci);
    unsigned out_h = U32(ci, OFF_OUTPUT_HEIGHT);
    while (U32(ci, OFF_OUTPUT_SCANLINE) < out_h) {
        uint8_t *rows[4];
        unsigned sl = U32(ci, OFF_OUTPUT_SCANLINE);
        for (int i = 0; i < 4; i++) rows[i] = out + (size_t)(sl + i < out_h ? sl + i : out_h - 1) * pitch;
        unsigned want = (out_h - sl) < 4 ? (out_h - sl) : 4;
        if (!L.read_scanlines(ci, rows, want)) break;
    }
    L.finish(ci);
    L.destroy(ci);
    return 0;
}

typedef struct {
    int n, mode, tid, nthreads, d;
    const uint8_t *const *datas;
    const size_t *lens;
    uint8_t *const *outs;
    const size_t *pitches;
    int rc;
} ScaledJob;

static void *scaled_worker(void *arg) {
    ScaledJob *j = (ScaledJob *)arg;
    for (int i = j->tid; i < j->n; i += j->nthreads) {
        int rc = decode_one_scaled(j->datas[i], j->lens[i], j->outs[i], j->pitches[i], j->mode, j->d);
        if (rc) j->rc = rc;
    }
    return NULL;
}

/* Decode n images at scale 1/d with `nthreads` host threads (round-robin assignment). */
int ljt_decode_batch_scaled(int n, const uint8_t *const *datas, const size_t *lens, uint8_t *const *outs,
                            const size_t *pitches, int mode, int nthreads, int d) {
    if (nthreads < 1) nthreads = 1;
    if (nthreads > n) nthreads = n;
    pthread_t *th = (pthread_t *)malloc(sizeof(pthread_t) * nthreads);
    ScaledJob *jobs = (ScaledJob *)malloc(sizeof(ScaledJob) * nthreads);
    int rc = 0;
    for (int t = 0; t < nthreads; t++) {
        jobs[t] = (ScaledJob){n, mode, t, nthreads, d, datas, lens, outs, pitches, 0};
        pthread_create(&th[t], NULL, scaled_worker, &jobs[t]);
    }
    for (int t = 0; t < nthreads; t++) {
        pthread_join(th[t], NULL);
        if (jobs[t].rc) rc = jobs[t].rc;
    }
    free(th);
    free(jobs);
    return rc;
}
