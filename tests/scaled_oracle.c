/* tests/scaled_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU restatement of the reduced-size decode
 * (HJD_FLAG_SCALE_*, include/hjd.h, DESIGN §2), the checker of csrc/scaled.cu.
 *
 * It is built on the plain-C restatement of the reference, oracle/jpeg_oracle.c, which it includes unchanged: the
 * header parse, the entropy decode, the IDCT constants and the colour conversion are that file's own functions.
 * tests/scaled_port.py compiles this file (with the oracle's flags: no contraction, no fast-math) into a library of
 * its own and binds it. */
#include "../oracle/jpeg_oracle.c"

/* ------------------------------------------------------------------ scaled ----------- */

/* DELIBERATE DEVIATION, no reference exists: reduced-size decode (the product's HJD_FLAG_SCALE_*, include/hjd.h).
   Every step is the reference's own step applied to the reduced block, so the result is exactly defined:
   de-quantisation as in hjdo_decode_single_block, then the direct-form IDCT of the top-left n x n natural-order
   coefficients with the cosine table of compute_idct_constants' expression with 16 replaced by 2n, then the colour
   step of hjdo_decode with 8 replaced by n.  With n = 8 this is hjdo_decode_single_block / hjdo_decode. */
static float g_cos_n[4][8][8];    /* [log2 n][p][k] = cosf(((2p+1) * k * PI) / (2n)), PI = 3.14f */
static int g_cos_n_ready[4];

static const float (*scaled_cos(int n))[8]
{
    const float PI = 3.14f;
    const int s = n == 8 ? 3 : (n == 4 ? 2 : (n == 2 ? 1 : 0));
    int p, k;
    if (!g_cos_n_ready[s]) {
        for (p = 0; p < n; p++)
            for (k = 0; k < n; k++) g_cos_n[s][p][k] = cosf(((2 * p + 1) * k * PI) / (float)(2 * n));
        g_cos_n_ready[s] = 1;
    }
    return (const float (*)[8])g_cos_n[s];
}

/* One block at n = 8, 4, 2 or 1 samples per side: n x n bytes at out (row stride `stride`); x horizontal. */
void hjdo_scaled_block(const int16_t coef[64], const float q[64], int n, uint8_t* out, int stride)
{
    int16_t data[64], block[64], arr[8][8];
    const float (*cs)[8];
    int c, i, x, y, u, v;
    init_tables();
    cs = scaled_cos(n);
    for (c = 0; c < 64; c++) data[c] = (int16_t)(int)(coef[c] * q[c]);           /* 150 */
    for (i = 0; i < 64; i++) block[i] = data[kZigZag[i]];                        /* 161 */
    for (y = 0, c = 0; y < 8; y++)
        for (x = 0; x < 8; x++) arr[x][y] = block[c++];                          /* 176 */
    for (y = 0; y < n; y++) {
        for (x = 0; x < n; x++) {
            float sum = 0;
            int16_t val;
            for (u = 0; u < n; u++)
                for (v = 0; v < n; v++)
                    sum += g_cc[u][v] * arr[u][v] * cs[x][u] * cs[y][v];         /* 120, n in place of 8 */
            val = (int16_t)(int)(0.25 * sum);                                    /* 123, 136 */
            val = (int16_t)(val + 128);                                          /* 137 */
            out[y * stride + x] = clamp_u8(val);                                 /* 219 */
        }
    }
}

/* Decode at 1 / 2^shift (shift 0..3) of the source size: rgb receives ceil(W / d) x ceil(H / d) RGB24 (d = 2^shift,
   libjpeg's jdiv_round_up).  Parse and entropy decode are hjdo_decode's; per MCU the luma tile is (n hF) x (n vF),
   the chroma tile n x n (Cb with Cr's table, 984), upsampled by the replication rule of 912 with 8 replaced by n. */
int hjdo_decode_scaled(const uint8_t* jpg, size_t size, int shift, uint8_t* rgb, unsigned* out_w, unsigned* out_h)
{
    frame_t* f;
    bits_t b;
    int rc, err = 0, c, n;
    int16_t prev_dc[4] = {0, 0, 0, 0};
    int16_t dct[64];
    uint8_t tY[256], tCb[64], tCr[64];
    unsigned hF, vF, xs, ys, d, ow, oh, x, y, mx, my, mcu = 0;
    if (shift < 0 || shift > 3) return HJDO_ERR_UNSUPPORTED;
    n = 8 >> shift;
    d = 1u << shift;
    f = (frame_t*)malloc(sizeof *f);
    if (!f) return HJDO_ERR_TRUNCATED;
    rc = parse_header(jpg, size, f);
    if (rc != HJDO_OK) { free(f); return rc; }
    ow = (f->width + d - 1) / d;
    oh = (f->height + d - 1) / d;
    if (out_w) *out_w = ow;
    if (out_h) *out_h = oh;
    init_tables();
    hF = f->ncomp == 3 ? f->hf[0] : 1;
    vF = f->ncomp == 3 ? f->vf[0] : 1;
    xs = 8 * hF; ys = 8 * vF;
    memset(&b, 0, sizeof b);
    b.s = f->scan; b.len = f->scan_len;
    memset(tCb, 128, 64); memset(tCr, 128, 64);

    for (y = 0, my = 0; y < f->height; y += ys, my++) {
        for (x = 0, mx = 0; x < f->width; x += xs, mx++, mcu++) {
            unsigned bx, by, px, py;
            if (f->restart_interval && mcu && mcu % (unsigned)f->restart_interval == 0) {
                if (stream_byte(&b, b.pos) != 0xFF || (stream_byte(&b, b.pos + 1) & 0xF8) != 0xD0) err = HJDO_ERR_RESTART;
                else b.pos += 2;
                b.reservoir = 0; b.nbits = 0;
                for (c = 0; c < 4; c++) prev_dc[c] = 0;
            }
            for (by = 0; by < vF; by++)
                for (bx = 0; bx < hF; bx++) {
                    int e = process_huffman_block(dct, &prev_dc[0], &f->dc[f->td[0]], &f->ac[f->ta[0]], &b);
                    if (e && !err) err = e;
                    hjdo_scaled_block(dct, f->q[f->tq[0]], n, &tY[bx * n + by * n * n * hF], (int)(n * hF));
                }
            if (f->ncomp == 3) {
                int e = process_huffman_block(dct, &prev_dc[1], &f->dc[f->td[1]], &f->ac[f->ta[1]], &b);
                if (e && !err) err = e;
                hjdo_scaled_block(dct, f->q[f->tq[2]], n, tCb, n);              /* 984: Cr's q-table (sic) */
                e = process_huffman_block(dct, &prev_dc[2], &f->dc[f->td[2]], &f->ac[f->ta[2]], &b);
                if (e && !err) err = e;
                hjdo_scaled_block(dct, f->q[f->tq[2]], n, tCr, n);
            }
            if (!rgb) continue;
            for (py = 0; py < n * vF; py++)
                for (px = 0; px < n * hF; px++) {
                    const unsigned ox = mx * n * hF + px, oy = my * n * vF + py;
                    int yoff, coff;
                    if (ox >= ow || oy >= oh) continue;
                    yoff = (int)(px + py * n * hF);
                    coff = (int)(px * (1.0f / hF)) + (int)(py * (1.0f / vF)) * n;   /* 912, n in place of 8 */
                    hjdo_ycc_to_rgb(tY[yoff], tCb[coff], tCr[coff], rgb + ((size_t)oy * ow + ox) * 3);
                }
        }
    }
    free(f);
    return err;
}

/* ------------------------------------------------------------------ loops for tests/colour_cube.py ----------- */

/* The colour step on every (Y, Cb, Cr) byte triple: rgb[((Y << 16) | (Cb << 8) | Cr) * 3 + channel], 48 MB.
   fma = 0: hjdo_ycc_to_rgb itself.  fma = 1: the same expressions with every product contracted into an FMA (what a
   compiler allowed to contract would make of them), so that the tests can count where contraction changes a byte. */
void hjdo_ycc_cube(int fma, uint8_t* rgb)
{
    int yc, cb, cr;
    for (yc = 0; yc < 256; yc++)
        for (cb = 0; cb < 256; cb++)
            for (cr = 0; cr < 256; cr++) {
                uint8_t* o = rgb + (((size_t)yc << 16) | ((size_t)cb << 8) | (size_t)cr) * 3;
                if (!fma) {
                    hjdo_ycc_to_rgb(yc, cb, cr, o);
                } else {
                    const float fy = (float)yc, fcb = (float)(cb - 128), fcr = (float)(cr - 128);
                    o[0] = clamp_u8((int)fmaf(1.402f, fcr, fy));
                    o[1] = clamp_u8((int)fmaf(-0.71414f, fcr, fmaf(-0.34414f, fcb, fy)));
                    o[2] = clamp_u8((int)fmaf(1.772f, fcb, fy));
                }
            }
}

/* The decoded sample of DC-only blocks (quantised DC c0[i], table entry q0[i] at the DC, every AC zero) through
   hjdo_decode_single_block (n = 8) or hjdo_scaled_block (n = 4, 2, 1): out[i].  Returns the number of samples that differ
   from the first sample of their block (a DC-only block decodes flat, so 0). */
long hjdo_dc_only(const int32_t* c0, const int32_t* q0, long count, int n, uint8_t* out)
{
    int16_t coef[64];
    float q[64];
    uint8_t blk[64];
    long i, uneven = 0;
    int k;
    memset(coef, 0, sizeof coef);
    for (k = 0; k < 64; k++) q[k] = 1.0f;
    for (i = 0; i < count; i++) {
        coef[0] = (int16_t)c0[i];
        q[0] = (float)q0[i];
        if (n == 8) hjdo_decode_single_block(coef, q, blk, 8);
        else hjdo_scaled_block(coef, q, n, blk, n);
        for (k = 1; k < n * n; k++) uneven += blk[k] != blk[0];
        out[i] = blk[0];
    }
    return uneven;
}
