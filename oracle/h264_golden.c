/*
 * ORACLE -- TEST INFRASTRUCTURE ONLY (see h264_golden.h for what is and is not pinned).
 *
 * Single-threaded, integer-only CPU golden model of the CQP I+P H.264 encoder.
 * Headers restate /root/reference/kernel/cedar.c (cited per function); slice data is our own
 * algorithm (the reference's is silicon) constrained by those headers and by H.264 decoder
 * conformance.  The CUDA product path must reproduce this model's output byte for byte.
 */
#include "h264_golden.h"
#include "h264_tables.h"

#include <errno.h>
#include <stdlib.h>
#include <string.h>

#define ALIGN(x, a) (((x) + ((a)-1)) & ~((a)-1))
#define CLIP3(lo, hi, v) ((v) < (lo) ? (lo) : ((v) > (hi) ? (hi) : (v)))
static inline int clip255(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); }
static inline int iabs(int v) { return v < 0 ? -v : v; }
static inline int imin(int a, int b) { return a < b ? a : b; }
static inline int imax(int a, int b) { return a > b ? a : b; }
static inline int me_lambda(int qp);

/* luma4x4BlkIdx <-> position inside the macroblock (in 4x4 units) */
static const uint8_t blk_x[16] = {0, 1, 0, 1, 2, 3, 2, 3, 0, 1, 0, 1, 2, 3, 2, 3};
static const uint8_t blk_y[16] = {0, 0, 1, 1, 0, 0, 1, 1, 2, 2, 3, 3, 2, 2, 3, 3};
static const uint8_t xy2blk[4][4] = {{0, 1, 4, 5}, {2, 3, 6, 7}, {8, 9, 12, 13}, {10, 11, 14, 15}}; /* [y][x] */

/* ------------------------------------------------------------------------------------------
 * Bit writer.  Restates cedar_bytestream_write / _expgolomb / _expgolomb_signed
 * (kernel/cedar.c:187-223): MSB-first append of <= 31 bits; ue(v) = v+1 in 2*bitlen-1 bits;
 * se(v): d = 2v-1; d ^= d>>31; ue(d).  The hardware PUTBITS port becomes a byte buffer.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    uint8_t *buf;
    size_t cap;
    size_t nbits;
} bitw;

static void bw_init(bitw *b, uint8_t *buf, size_t cap)
{
    b->buf = buf;
    b->cap = cap;
    b->nbits = 0;
}

static void bw_put(bitw *b, uint32_t data, int size)
{
    for (int i = size - 1; i >= 0; i--) {
        size_t byte = b->nbits >> 3;
        if (byte >= b->cap)
            return; /* overflow: caller checks nbits against cap */
        int bit = (data >> i) & 1;
        if ((b->nbits & 7) == 0)
            b->buf[byte] = 0;
        b->buf[byte] |= bit << (7 - (b->nbits & 7));
        b->nbits++;
    }
}

static __attribute__((unused)) int ue_len(uint32_t v)
{
    v++;
    return (32 - __builtin_clz(v)) * 2 - 1;
}

static void bw_ue(bitw *b, uint32_t v) /* cedar.c:209-215 */
{
    v++;
    bw_put(b, v, (32 - __builtin_clz(v)) * 2 - 1);
}

static void bw_se(bitw *b, int32_t v) /* cedar.c:217-223 */
{
    v = (2 * v) - 1;
    v ^= (v >> 31);
    bw_ue(b, (uint32_t)v);
}

/* cedar.c:883-890.  len = bits in the stream so far (STMLEN); every NAL starts byte aligned so
 * only len & 7 matters.  Quirk kept: with 7 bits used in the last byte, pad = 8 and nine bits
 * (the stop bit and a whole 0x00 byte) are written. */
static void bw_trailing_cedar(bitw *b)
{
    uint32_t len = (uint32_t)b->nbits;
    int pad = 8 - ((len + 1) & 0x7);
    bw_put(b, 1u << pad, pad + 1);
}

/* Emulation prevention (done by the VE hardware in the reference, toggled off only for the
 * start code, cedar.c:872-880): insert 0x03 after 00 00 when the next byte is <= 3. */
static size_t epb_copy(uint8_t *dst, size_t cap, const uint8_t *src, size_t n)
{
    size_t o = 0;
    int zeros = 0;
    for (size_t i = 0; i < n; i++) {
        if (zeros >= 2 && src[i] <= 3) {
            if (o < cap)
                dst[o] = 3;
            o++;
            zeros = 0;
        }
        if (o < cap)
            dst[o] = src[i];
        o++;
        zeros = src[i] == 0 ? zeros + 1 : 0;
    }
    return o;
}

/* cedar.c:868-881: 24 zero bits, then 16 bits 0x0100 | ref_idc<<5 | type  => 00 00 00 01 hh */
static size_t put_startcode(uint8_t *out, int ref_idc, int type)
{
    out[0] = 0;
    out[1] = 0;
    out[2] = 0;
    out[3] = 1;
    out[4] = (uint8_t)(((ref_idc & 3) << 5) | (type & 0x1f));
    return 5;
}

/* cedar.c:892-937 */
int gm_write_sps(const gm_config *cfg, uint8_t *out, int cap)
{
    uint8_t rb[64];
    bitw b;
    int w_mb = ALIGN(cfg->dst_width, 16) >> 4, h_mb = ALIGN(cfg->dst_height, 16) >> 4;
    bw_init(&b, rb, sizeof(rb));
    bw_put(&b, (uint32_t)cfg->profile, 8);
    bw_put(&b, 0, 8); /* constraints */
    {
        /* auto_level extension: lowest level whose MaxFS (table A-1) holds the picture; cedar.c:900 writes cfg->level */
        static const int max_fs[][2] = {{99, 10},   {396, 11},  {792, 21},   {1620, 22},  {3600, 31},  {5120, 32},
                                        {8192, 40}, {8704, 42}, {22080, 50}, {36864, 51}, {139264, 60}};
        int level = cfg->level;
        if (cfg->auto_level) {
            level = 62;
            for (int i = 10; i >= 0; i--)
                if (w_mb * h_mb <= max_fs[i][0])
                    level = max_fs[i][1];
        }
        bw_put(&b, (uint32_t)level, 8);
    }
    bw_ue(&b, 0); /* seq_parameter_set_id */
    bw_ue(&b, 0); /* log2_max_frame_num_minus4 */
    bw_ue(&b, 2); /* pic_order_cnt_type */
    bw_ue(&b, 1); /* max_num_ref_frames */
    bw_put(&b, 0, 1); /* gaps_in_frame_num_value_allowed_flag */
    bw_ue(&b, (uint32_t)(w_mb - 1));
    bw_ue(&b, (uint32_t)(h_mb - 1));
    bw_put(&b, 1, 1); /* frame_mbs_only_flag */
    bw_put(&b, 0, 1); /* direct_8x8_inference_flag */
    if (cfg->sps_crop && (w_mb * 16 > cfg->src_width || h_mb * 16 > cfg->src_height)) {
        /* sps_crop extension, field order of cedar.c:924-929; offsets in crop units of two luma samples */
        bw_put(&b, 1, 1);
        bw_ue(&b, 0);
        bw_ue(&b, (uint32_t)((w_mb * 16 - cfg->src_width) / 2));
        bw_ue(&b, 0);
        bw_ue(&b, (uint32_t)((h_mb * 16 - cfg->src_height) / 2));
    } else
        bw_put(&b, 0, 1); /* frame_cropping_flag: crop is always 0 (cedar.c:756-761 makes :924-931 dead) */
    bw_put(&b, 0, 1); /* vui_parameters_present_flag */
    bw_trailing_cedar(&b);
    if (cap < 5 + 2 * (int)(b.nbits >> 3))
        return -ENOMEM;
    size_t n = put_startcode(out, 3, 7);
    n += epb_copy(out + n, (size_t)cap - n, rb, b.nbits >> 3);
    return (int)n;
}

/* cedar.c:939-982 */
int gm_write_pps(const gm_config *cfg, uint8_t *out, int cap)
{
    uint8_t rb[64];
    bitw b;
    bw_init(&b, rb, sizeof(rb));
    bw_ue(&b, 0); /* pic_parameter_set_id */
    bw_ue(&b, 0); /* seq_parameter_set_id */
    bw_put(&b, cfg->entropy_coding_mode == GM_ENTROPY_CABAC ? 1 : 0, 1);
    bw_put(&b, 0, 1); /* bottom_field_pic_order_in_frame_present_flag */
    bw_ue(&b, 0);     /* num_slice_groups_minus1 */
    bw_ue(&b, 0);     /* num_ref_idx_l0_default_active_minus1 */
    bw_ue(&b, 0);     /* num_ref_idx_l1_default_active_minus1 */
    bw_put(&b, 0, 1); /* weighted_pred_flag */
    bw_put(&b, 0, 2); /* weighted_bipred_idc */
    bw_se(&b, cfg->qp - 26);
    bw_se(&b, cfg->qp - 26);
    bw_se(&b, 4);     /* chroma_qp_index_offset */
    bw_put(&b, 1, 1); /* deblocking_filter_control_present_flag */
    bw_put(&b, 0, 1); /* constrained_intra_pred_flag */
    bw_put(&b, 0, 1); /* redundant_pic_cnt_present_flag */
    bw_trailing_cedar(&b);
    if (cap < 5 + 2 * (int)(b.nbits >> 3))
        return -ENOMEM;
    size_t n = put_startcode(out, 3, 8);
    n += epb_copy(out + n, (size_t)cap - n, rb, b.nbits >> 3);
    return (int)n;
}

/* cedar.c:984-1030 (bits after the NAL header byte) */
static void write_slice_header(bitw *b, int frame_i, int frame_p_count, int cabac, int first_mb)
{
    bw_ue(b, (uint32_t)first_mb); /* first_mb_in_slice: 0 in the reference (cedar.c:992-993, one slice per picture) */
    bw_ue(b, frame_i ? 2 : 0);  /* slice_type */
    bw_ue(b, 0);                /* pic_parameter_set_id */
    bw_put(b, (uint32_t)frame_p_count & 0x0F, 4); /* frame_num */
    if (frame_i) {
        bw_ue(b, 0);     /* idr_pic_id */
        bw_put(b, 0, 1); /* no_output_of_prior_pics_flag */
        bw_put(b, 0, 1); /* long_term_reference_flag */
    } else {
        bw_put(b, 0, 1); /* num_ref_idx_active_override_flag */
        bw_put(b, 0, 1); /* ref_pic_list_modification_flag_l0 */
        bw_put(b, 0, 1); /* adaptive_ref_pic_marking_mode_flag */
        if (cabac)
            bw_ue(b, 0); /* cabac_init_idc */
    }
    bw_se(b, 0); /* slice_qp_delta */
    bw_ue(b, 0); /* disable_deblocking_filter_idc */
    bw_se(b, 0); /* slice_alpha_c0_offset_div2 */
    bw_se(b, 0); /* slice_beta_offset_div2 */
}

int gm_slice_header_bits64(int frame_i, int frame_p_count, int cabac, int first_mb, uint64_t *bits, int *nbits)
{
    uint8_t rb[16] = {0};
    bitw b;
    bw_init(&b, rb, sizeof(rb));
    write_slice_header(&b, frame_i, frame_p_count, cabac, first_mb);
    *nbits = (int)b.nbits;
    uint64_t v = 0;
    for (int i = 0; i < 8; i++)
        v = (v << 8) | rb[i];
    *bits = v >> (64 - b.nbits);
    return 0;
}

int gm_slice_header_bits(int frame_i, int frame_p_count, int cabac, uint32_t *bits, int *nbits)
{
    uint64_t v;
    gm_slice_header_bits64(frame_i, frame_p_count, cabac, 0, &v, nbits);
    *bits = (uint32_t)v;
    return 0;
}

/* ------------------------------------------------------------------------------------------
 * Synthetic clip
 * ------------------------------------------------------------------------------------------ */
static inline int tri256(int v)
{
    v &= 255;
    return v < 128 ? v : 255 - v;
}

void gm_synth_frame(int width, int height, int format, int t, uint8_t *luma, uint8_t *chroma)
{
    int fx = ((100 - 5 * t) % width + width) % width;
    int fy = ((60 + 4 * t) % height + height) % height;
    for (int y = 0; y < height; y++)
        for (int x = 0; x < width; x++) {
            int xs = x + 3 * t, ys = y + 2 * t;
            int v = 40 + (tri256(xs * 2 + ys) >> 1) + ((((xs >> 3) ^ (ys >> 3)) & 7) * 6) + (((xs * ys) >> 6) & 7);
            int rx = x - fx, ry = y - fy;
            if (rx < 0)
                rx += width;
            if (ry < 0)
                ry += height;
            if (rx < 128 && ry < 128)
                v = 200 - (tri256(rx * 4 + ry * 2) >> 1) + ((rx ^ ry) & 15);
            uint32_t h = (uint32_t)x * 0x9E3779B1u + (uint32_t)y * 0x85EBCA77u + (uint32_t)t * 0xC2B2AE3Du;
            h ^= h >> 15;
            h *= 0x2C1B3C6Du;
            h ^= h >> 12;
            v += (int)((h >> 8) % 5u) - 2;
            luma[(size_t)y * width + x] = (uint8_t)clip255(v);
        }
    int crows = format == GM_FORMAT_NV16 ? height : height / 2;
    for (int r = 0; r < crows; r++) {
        int cy = format == GM_FORMAT_NV16 ? (r >> 1) : r;
        for (int cx = 0; cx < width / 2; cx++) {
            chroma[(size_t)r * width + 2 * cx] = (uint8_t)(128 + ((cx + t) & 63) - 32);
            chroma[(size_t)r * width + 2 * cx + 1] = (uint8_t)(128 + ((cy + 2 * t) & 63) - 32);
        }
    }
}

/* ------------------------------------------------------------------------------------------
 * Encoder state (mirrors struct sunxi_cedar's encode fields, kernel/cedar.c:75-134)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    uint8_t *p[3]; /* Y, U, V planar; strides W, W/2, W/2 */
} frame_t;

struct gm_encoder {
    gm_config cfg;
    int W, H, mbw, mbh;
    int srows; /* macroblock rows per slice (mbh = one slice per picture, the reference's layout) */
    int qp, qpc;
    int frame_p_count, frame_count; /* cedar.c:118-119 counters */
    frame_t src, rec[2], unf;
    int cur;                        /* reference_current index (ping-pong, cedar.c:1198-1201) */
    gm_mb *mbs;
    uint8_t *refpad; /* edge-extended reference luma for the motion search */
    uint32_t *inter_cost; /* p_intra: best motion-search cost (SAD + lambda * mv bits) per macroblock */
    uint8_t *want_intra;  /* p_intra: decision per macroblock */
    uint8_t *rbsp;
    size_t rbsp_cap;
    int last_frame_i;
    double last_sse_y;
};

static int frame_alloc(frame_t *f, int W, int H)
{
    f->p[0] = (uint8_t *)calloc((size_t)W * H, 1);
    f->p[1] = (uint8_t *)calloc((size_t)W * H / 4, 1);
    f->p[2] = (uint8_t *)calloc((size_t)W * H / 4, 1);
    return f->p[0] && f->p[1] && f->p[2] ? 0 : -ENOMEM;
}

static void frame_free(frame_t *f)
{
    for (int i = 0; i < 3; i++)
        free(f->p[i]);
}

/* cedar.c:744-789 validation, same order and same -EINVAL */
int gm_open(const gm_config *cfg, gm_encoder **out)
{
    if (!cfg || !out)
        return -EINVAL;
    if ((cfg->src_width & 1) || (cfg->src_height & 1))
        return -EINVAL;
    if ((cfg->dst_width & 0x0F) || (cfg->dst_height & 0x0F))
        return -EINVAL;
    if (cfg->src_width > cfg->dst_width || cfg->src_height > cfg->dst_height)
        return -EINVAL;
    if (cfg->qp <= 0 || cfg->qp > 47)
        return -EINVAL;
    if (cfg->src_format != GM_FORMAT_NV12 && cfg->src_format != GM_FORMAT_NV16)
        return -EINVAL;
    if (cfg->keyframe_interval <= 0 || (cfg->keyframe_interval >= 32 && !cfg->relax_gop))
        return -EINVAL;
    if (cfg->src_width <= 0 || cfg->src_height <= 0 || cfg->me_range < 0 || cfg->me_range > 64 || cfg->slice_rows < 0)
        return -EINVAL;

    gm_encoder *e = (gm_encoder *)calloc(1, sizeof(*e));
    if (!e)
        return -ENOMEM;
    e->cfg = *cfg;
    if (e->cfg.me_range == 0)
        e->cfg.me_range = 16;
    e->W = cfg->dst_width;
    e->H = cfg->dst_height;
    e->mbw = e->W >> 4;
    e->mbh = e->H >> 4;
    e->srows = cfg->slice_rows > 0 && cfg->slice_rows < e->mbh ? cfg->slice_rows : e->mbh;
    e->qp = cfg->qp;
    e->qpc = h264_chroma_qp[CLIP3(0, 51, cfg->qp + 4)]; /* chroma_qp_index_offset = 4, cedar.c:969 */
    int err = frame_alloc(&e->src, e->W, e->H) | frame_alloc(&e->rec[0], e->W, e->H) |
              frame_alloc(&e->rec[1], e->W, e->H) | frame_alloc(&e->unf, e->W, e->H);
    e->mbs = (gm_mb *)calloc((size_t)e->mbw * e->mbh, sizeof(gm_mb));
    e->inter_cost = (uint32_t *)calloc((size_t)e->mbw * e->mbh, sizeof(uint32_t));
    e->want_intra = (uint8_t *)calloc((size_t)e->mbw * e->mbh, 1);
    e->rbsp_cap = (size_t)e->mbw * e->mbh * 2048 + 4096;
    e->rbsp = (uint8_t *)malloc(e->rbsp_cap);
    if (err || !e->mbs || !e->rbsp) {
        gm_close(e);
        return -ENOMEM;
    }
    *out = e;
    return 0;
}

void gm_close(gm_encoder *e)
{
    if (!e)
        return;
    frame_free(&e->src);
    frame_free(&e->rec[0]);
    frame_free(&e->rec[1]);
    frame_free(&e->unf);
    free(e->mbs);
    free(e->refpad);
    free(e->inter_cost);
    free(e->want_intra);
    free(e->rbsp);
    free(e);
}

/* Is the macroblock row above row mby in the same slice?  Slices are whole macroblock rows, so the left
 * neighbour always is; neighbours in other slices are "not available" (H.264 6.4.x) for intra prediction,
 * motion-vector prediction and every entropy-coding context -- but not for the deblocking filter, which runs
 * across slice edges when disable_deblocking_filter_idc = 0 (cedar.c:1025). */
static inline int top_avail(const gm_encoder *e, int mby) { return (mby % e->srows) != 0; }

int gm_coded_width(const gm_encoder *e) { return e->W; }
int gm_coded_height(const gm_encoder *e) { return e->H; }
const gm_mb *gm_mbs(const gm_encoder *e) { return e->mbs; }
const uint8_t *gm_recon(const gm_encoder *e, int plane) { return e->rec[e->cur ^ 1].p[plane]; }
const uint8_t *gm_recon_unfiltered(const gm_encoder *e, int plane) { return e->unf.p[plane]; }
const uint8_t *gm_source(const gm_encoder *e, int plane) { return e->src.p[plane]; }
int gm_last_frame_type(const gm_encoder *e) { return e->last_frame_i; }
double gm_last_sse_y(const gm_encoder *e) { return e->last_sse_y; }
void gm_set_frame_p_count(gm_encoder *e, int frame_p_count) { e->frame_p_count = frame_p_count; }

/* ------------------------------------------------------------------------------------------
 * K0 ingest: packed w x h NV12/NV16 -> planar 4:2:0 at the coded size, edge replicated.
 * NV16 -> 4:2:0: rounding average of the two chroma rows (SURVEY M5; unpinned by the reference,
 * which validates NV16 at cedar.c:777-782 and then never reads the format again).
 * ------------------------------------------------------------------------------------------ */
static void ingest(gm_encoder *e, const uint8_t *luma, const uint8_t *chroma)
{
    int w = e->cfg.src_width, h = e->cfg.src_height, W = e->W, H = e->H;
    for (int y = 0; y < H; y++) {
        int sy = imin(y, h - 1);
        for (int x = 0; x < W; x++)
            e->src.p[0][(size_t)y * W + x] = luma[(size_t)sy * w + imin(x, w - 1)];
    }
    int cw = w / 2, ch = h / 2, CW = W / 2, CH = H / 2;
    for (int y = 0; y < CH; y++) {
        int sy = imin(y, ch - 1);
        for (int x = 0; x < CW; x++) {
            int sx = imin(x, cw - 1);
            for (int c = 0; c < 2; c++) {
                int v;
                if (e->cfg.src_format == GM_FORMAT_NV16) {
                    int a = chroma[(size_t)(2 * sy) * w + 2 * sx + c];
                    int b = chroma[(size_t)(2 * sy + 1) * w + 2 * sx + c];
                    v = (a + b + 1) >> 1;
                } else
                    v = chroma[(size_t)sy * w + 2 * sx + c];
                e->src.p[1 + c][(size_t)y * CW + x] = (uint8_t)v;
            }
        }
    }
}

/* ------------------------------------------------------------------------------------------
 * Transform / quantisation (4x4 integer transform only; flat scaling lists)
 * ------------------------------------------------------------------------------------------ */
static inline int pos_class(int i) /* raster index 0..15 -> 0 (a), 1 (b), 2 (c) */
{
    int r = i >> 2, c = i & 3;
    if (!(r & 1) && !(c & 1))
        return 0;
    if ((r & 1) && (c & 1))
        return 1;
    return 2;
}

static void fdct4x4(const int16_t *d /* raster 4x4 residual */, int *w)
{
    int t[16];
    for (int i = 0; i < 4; i++) { /* rows */
        int a = d[i * 4 + 0], b = d[i * 4 + 1], c = d[i * 4 + 2], e = d[i * 4 + 3];
        int s03 = a + e, d03 = a - e, s12 = b + c, d12 = b - c;
        t[i * 4 + 0] = s03 + s12;
        t[i * 4 + 1] = 2 * d03 + d12;
        t[i * 4 + 2] = s03 - s12;
        t[i * 4 + 3] = d03 - 2 * d12;
    }
    for (int i = 0; i < 4; i++) { /* columns */
        int a = t[i], b = t[4 + i], c = t[8 + i], e = t[12 + i];
        int s03 = a + e, d03 = a - e, s12 = b + c, d12 = b - c;
        w[i] = s03 + s12;
        w[4 + i] = 2 * d03 + d12;
        w[8 + i] = s03 - s12;
        w[12 + i] = d03 - 2 * d12;
    }
}

/* Inverse 4x4 transform of already-scaled coefficients, rows first then columns, (x+32)>>6. */
static void idct4x4_add(const int *d, uint8_t *dst, int stride, const uint8_t *pred, int pstride)
{
    int t[16];
    for (int i = 0; i < 4; i++) {
        int d0 = d[i * 4], d1 = d[i * 4 + 1], d2 = d[i * 4 + 2], d3 = d[i * 4 + 3];
        int e0 = d0 + d2, e1 = d0 - d2, e2 = (d1 >> 1) - d3, e3 = d1 + (d3 >> 1);
        t[i * 4 + 0] = e0 + e3;
        t[i * 4 + 1] = e1 + e2;
        t[i * 4 + 2] = e1 - e2;
        t[i * 4 + 3] = e0 - e3;
    }
    for (int i = 0; i < 4; i++) {
        int d0 = t[i], d1 = t[4 + i], d2 = t[8 + i], d3 = t[12 + i];
        int e0 = d0 + d2, e1 = d0 - d2, e2 = (d1 >> 1) - d3, e3 = d1 + (d3 >> 1);
        int r0 = e0 + e3, r1 = e1 + e2, r2 = e1 - e2, r3 = e0 - e3;
        dst[0 * stride + i] = (uint8_t)clip255(pred[0 * pstride + i] + ((r0 + 32) >> 6));
        dst[1 * stride + i] = (uint8_t)clip255(pred[1 * pstride + i] + ((r1 + 32) >> 6));
        dst[2 * stride + i] = (uint8_t)clip255(pred[2 * pstride + i] + ((r2 + 32) >> 6));
        dst[3 * stride + i] = (uint8_t)clip255(pred[3 * pstride + i] + ((r3 + 32) >> 6));
    }
}

static inline int quant1(int w, int mf, int f, int shift)
{
    int a = (iabs(w) * mf + f) >> shift;
    return w < 0 ? -a : a;
}

static inline int dequant_ac(int c, int qp, int cls)
{
    int ls = 16 * h264_dequant_v[qp % 6][cls];
    if (qp >= 24)
        return (c * ls) * (1 << (qp / 6 - 4));
    return (c * ls + (1 << (3 - qp / 6))) >> (4 - qp / 6);
}

/* Quantise a transformed block into zig-zag levels [first..15]; returns non-zero count. */
static int quant_block(const int *w, int qp, int intra, int first, int16_t *lev)
{
    int qbits = 15 + qp / 6;
    int f = (1 << qbits) / (intra ? 3 : 6);
    int nnz = 0;
    for (int i = 0; i < first; i++)
        lev[i] = 0;
    for (int i = first; i < 16; i++) {
        int r = h264_zigzag4x4[i];
        int z = quant1(w[r], h264_quant_mf[qp % 6][pos_class(r)], f, qbits);
        lev[i] = (int16_t)z;
        nnz += z != 0;
    }
    return nnz;
}

/* Residual of one 4x4 block */
static void resid4x4(const uint8_t *src, int sstride, const uint8_t *pred, int pstride, int16_t *d)
{
    for (int y = 0; y < 4; y++)
        for (int x = 0; x < 4; x++)
            d[y * 4 + x] = (int16_t)(src[y * sstride + x] - pred[y * pstride + x]);
}

/* Dequantise levels (zig-zag, from index `first`) into raster coefficient array; dc preset by caller */
static void dequant_block(const int16_t *lev, int qp, int first, int *d)
{
    for (int i = first; i < 16; i++) {
        int r = h264_zigzag4x4[i];
        d[r] = dequant_ac(lev[i], qp, pos_class(r));
    }
}

/* Chroma of one macroblock (both planes): transform, DC Hadamard, quant, recon.  Shared by
 * intra and inter.  pred = 8x8 prediction per plane (stride 8). */
static void encode_chroma(gm_encoder *e, gm_mb *mb, int mbx, int mby, const uint8_t pred[2][64], int intra,
                          frame_t *out)
{
    int CW = e->W / 2, qpc = e->qpc;
    int qbits = 15 + qpc / 6, f = (1 << qbits) / (intra ? 3 : 6);
    int any_dc = 0, any_ac = 0;
    int wblk[2][4][16];
    for (int c = 0; c < 2; c++) {
        const uint8_t *src = e->src.p[1 + c] + (size_t)(mby * 8) * CW + mbx * 8;
        int dc[4];
        for (int b = 0; b < 4; b++) {
            int bx = (b & 1) * 4, by = (b >> 1) * 4;
            int16_t d[16];
            resid4x4(src + by * CW + bx, CW, pred[c] + by * 8 + bx, 8, d);
            fdct4x4(d, wblk[c][b]);
            dc[b] = wblk[c][b][0];
            int n = quant_block(wblk[c][b], qpc, intra, 1, mb->coef[18 + c * 4 + b]);
            mb->nnz[17 + c * 4 + b] = (uint8_t)n;
            any_ac |= n;
        }
        /* 2x2 Hadamard, |Z| = (|Y|*MF0 + 2f) >> (qbits+1) */
        int y0 = dc[0] + dc[1] + dc[2] + dc[3], y1 = dc[0] - dc[1] + dc[2] - dc[3];
        int y2 = dc[0] + dc[1] - dc[2] - dc[3], y3 = dc[0] - dc[1] - dc[2] + dc[3];
        int yd[4] = {y0, y1, y2, y3};
        int n = 0;
        for (int i = 0; i < 4; i++) {
            int z = quant1(yd[i], h264_quant_mf[qpc % 6][0], 2 * f, qbits + 1);
            mb->coef[17][c * 4 + i] = (int16_t)z;
            n += z != 0;
        }
        mb->nnz[25 + c] = (uint8_t)n;
        any_dc |= n;
    }
    int cbpc = any_ac ? 2 : (any_dc ? 1 : 0);
    mb->cbp = (uint8_t)((mb->cbp & 15) | (cbpc << 4));
    if (cbpc < 2)
        for (int i = 17; i <= 24; i++)
            mb->nnz[i] = 0;
    if (cbpc < 1)
        mb->nnz[25] = mb->nnz[26] = 0;
    /* reconstruction: exactly what a decoder does with the signalled levels */
    for (int c = 0; c < 2; c++) {
        uint8_t *dst = out->p[1 + c] + (size_t)(mby * 8) * CW + mbx * 8;
        int dcq[4] = {0, 0, 0, 0};
        if (cbpc >= 1) {
            const int16_t *z = &mb->coef[17][c * 4];
            int f0 = z[0] + z[1] + z[2] + z[3], f1 = z[0] - z[1] + z[2] - z[3];
            int f2 = z[0] + z[1] - z[2] - z[3], f3 = z[0] - z[1] - z[2] + z[3];
            int ls = 16 * h264_dequant_v[qpc % 6][0];
            dcq[0] = ((f0 * ls) * (1 << (qpc / 6))) >> 5;
            dcq[1] = ((f1 * ls) * (1 << (qpc / 6))) >> 5;
            dcq[2] = ((f2 * ls) * (1 << (qpc / 6))) >> 5;
            dcq[3] = ((f3 * ls) * (1 << (qpc / 6))) >> 5;
        }
        for (int b = 0; b < 4; b++) {
            int bx = (b & 1) * 4, by = (b >> 1) * 4;
            int d[16] = {0};
            if (cbpc == 2)
                dequant_block(mb->coef[18 + c * 4 + b], qpc, 1, d);
            d[0] = dcq[b];
            idct4x4_add(d, dst + by * CW + bx, CW, pred[c] + by * 8 + bx, 8);
        }
    }
}

/* ------------------------------------------------------------------------------------------
 * K4 intra (I frames): Intra16x16 V/H/DC/Plane by SAD, chroma DC/H/V/Plane by SAD.
 * Neighbours are the UNFILTERED reconstruction of left/top/top-left macroblocks.
 * ------------------------------------------------------------------------------------------ */
static void pred16x16(int mode, const uint8_t *top, const uint8_t *left, int tl, int has_top, int has_left,
                      uint8_t *pred)
{
    if (mode == 0) {
        for (int y = 0; y < 16; y++)
            memcpy(pred + y * 16, top, 16);
    } else if (mode == 1) {
        for (int y = 0; y < 16; y++)
            memset(pred + y * 16, left[y], 16);
    } else if (mode == 2) {
        int s = 0, dc;
        if (has_top)
            for (int i = 0; i < 16; i++)
                s += top[i];
        if (has_left)
            for (int i = 0; i < 16; i++)
                s += left[i];
        if (has_top && has_left)
            dc = (s + 16) >> 5;
        else if (has_top || has_left)
            dc = (s + 8) >> 4;
        else
            dc = 128;
        memset(pred, dc, 256);
    } else {
        int Hh = 0, Vv = 0;
        for (int i = 0; i < 8; i++) {
            int tm = i == 7 ? tl : top[6 - i];
            int lm = i == 7 ? tl : left[6 - i];
            Hh += (i + 1) * (top[8 + i] - tm);
            Vv += (i + 1) * (left[8 + i] - lm);
        }
        int a = 16 * (left[15] + top[15]);
        int b = (5 * Hh + 32) >> 6, c = (5 * Vv + 32) >> 6;
        for (int y = 0; y < 16; y++)
            for (int x = 0; x < 16; x++)
                pred[y * 16 + x] = (uint8_t)clip255((a + b * (x - 7) + c * (y - 7) + 16) >> 5);
    }
}

static void pred_chroma8x8(int mode, const uint8_t *top, const uint8_t *left, int tl, int has_top, int has_left,
                           uint8_t *pred)
{
    if (mode == 0) { /* DC, per 4x4 block */
        for (int b = 0; b < 4; b++) {
            int bx = b & 1, by = b >> 1;
            int st = 0, sl = 0, dc;
            for (int i = 0; i < 4; i++) {
                st += has_top ? top[bx * 4 + i] : 0;
                sl += has_left ? left[by * 4 + i] : 0;
            }
            int use_t = has_top, use_l = has_left;
            if (bx == 1 && by == 0 && has_top)
                use_l = 0; /* top-right block prefers top */
            if (bx == 0 && by == 1 && has_left)
                use_t = 0; /* bottom-left block prefers left */
            if (use_t && use_l)
                dc = (st + sl + 4) >> 3;
            else if (use_t)
                dc = (st + 2) >> 2;
            else if (use_l)
                dc = (sl + 2) >> 2;
            else
                dc = 128;
            for (int y = 0; y < 4; y++)
                memset(pred + (by * 4 + y) * 8 + bx * 4, dc, 4);
        }
    } else if (mode == 1) {
        for (int y = 0; y < 8; y++)
            memset(pred + y * 8, left[y], 8);
    } else if (mode == 2) {
        for (int y = 0; y < 8; y++)
            memcpy(pred + y * 8, top, 8);
    } else {
        int Hh = 0, Vv = 0;
        for (int i = 0; i < 4; i++) {
            int tm = i == 3 ? tl : top[2 - i];
            int lm = i == 3 ? tl : left[2 - i];
            Hh += (i + 1) * (top[4 + i] - tm);
            Vv += (i + 1) * (left[4 + i] - lm);
        }
        int a = 16 * (left[7] + top[7]);
        int b = (34 * Hh + 32) >> 6, c = (34 * Vv + 32) >> 6;
        for (int y = 0; y < 8; y++)
            for (int x = 0; x < 8; x++)
                pred[y * 8 + x] = (uint8_t)clip255((a + b * (x - 3) + c * (y - 3) + 16) >> 5);
    }
}

static int sad_block(const uint8_t *a, int as, const uint8_t *b, int bs, int w, int h)
{
    int s = 0;
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++)
            s += iabs(a[y * as + x] - b[y * bs + x]);
    return s;
}


/* ------------------------------------------------------------------------------------------
 * Intra4x4 (H.264 8.3.1): nine prediction modes from the reconstructed neighbours of each 4x4
 * block, blocks coded in luma4x4BlkIdx order.  edge layout: t[0..7] = A..H (above, above-right),
 * l[0..3] = I..L (left), m = M (above-left).
 * ------------------------------------------------------------------------------------------ */
static void pred4x4(int mode, const int *t, const int *l, int m, int has_top, int has_left, uint8_t *pred /* 16 */)
{
#define PT(x) ((x) < 0 ? m : t[x])
#define PL(y) ((y) < 0 ? m : l[y])
    for (int y = 0; y < 4; y++)
        for (int x = 0; x < 4; x++) {
            int v;
            switch (mode) {
            case 0: v = t[x]; break;
            case 1: v = l[y]; break;
            case 2: {
                int s = 0;
                if (has_top)
                    s += t[0] + t[1] + t[2] + t[3];
                if (has_left)
                    s += l[0] + l[1] + l[2] + l[3];
                v = (has_top && has_left) ? (s + 4) >> 3 : ((has_top || has_left) ? (s + 2) >> 2 : 128);
                break;
            }
            case 3: /* diagonal down left */
                v = (x == 3 && y == 3) ? (t[6] + 3 * t[7] + 2) >> 2 : (t[x + y] + 2 * t[x + y + 1] + t[x + y + 2] + 2) >> 2;
                break;
            case 4: /* diagonal down right */
                if (x > y)
                    v = (PT(x - y - 2) + 2 * PT(x - y - 1) + PT(x - y) + 2) >> 2;
                else if (x < y)
                    v = (PL(y - x - 2) + 2 * PL(y - x - 1) + PL(y - x) + 2) >> 2;
                else
                    v = (t[0] + 2 * m + l[0] + 2) >> 2;
                break;
            case 5: { /* vertical right */
                int z = 2 * x - y;
                if (z >= 0 && !(z & 1))
                    v = (PT(x - (y >> 1) - 1) + PT(x - (y >> 1)) + 1) >> 1;
                else if (z >= 0)
                    v = (PT(x - (y >> 1) - 2) + 2 * PT(x - (y >> 1) - 1) + PT(x - (y >> 1)) + 2) >> 2;
                else if (z == -1)
                    v = (l[0] + 2 * m + t[0] + 2) >> 2;
                else
                    v = (PL(y - 1) + 2 * PL(y - 2) + PL(y - 3) + 2) >> 2;
                break;
            }
            case 6: { /* horizontal down */
                int z = 2 * y - x;
                if (z >= 0 && !(z & 1))
                    v = (PL(y - (x >> 1) - 1) + PL(y - (x >> 1)) + 1) >> 1;
                else if (z >= 0)
                    v = (PL(y - (x >> 1) - 2) + 2 * PL(y - (x >> 1) - 1) + PL(y - (x >> 1)) + 2) >> 2;
                else if (z == -1)
                    v = (l[0] + 2 * m + t[0] + 2) >> 2;
                else
                    v = (PT(x - 1) + 2 * PT(x - 2) + PT(x - 3) + 2) >> 2;
                break;
            }
            case 7: /* vertical left */
                if (!(y & 1))
                    v = (t[x + (y >> 1)] + t[x + (y >> 1) + 1] + 1) >> 1;
                else
                    v = (t[x + (y >> 1)] + 2 * t[x + (y >> 1) + 1] + t[x + (y >> 1) + 2] + 2) >> 2;
                break;
            default: { /* 8: horizontal up */
                int z = x + 2 * y;
                if (z > 5)
                    v = l[3];
                else if (z == 5)
                    v = (l[2] + 3 * l[3] + 2) >> 2;
                else if (!(z & 1))
                    v = (l[y + (x >> 1)] + l[y + (x >> 1) + 1] + 1) >> 1;
                else
                    v = (l[y + (x >> 1)] + 2 * l[y + (x >> 1) + 1] + l[y + (x >> 1) + 2] + 2) >> 2;
                break;
            }
            }
            pred[y * 4 + x] = (uint8_t)v;
        }
#undef PT
#undef PL
}

/* Intra4x4PredMode of the 4x4 block left of / above block blk of macroblock (mbx, mby) for the
 * prediction of the mode: -1 = not available (=> predicted mode 2), 2 when the neighbour MB is
 * not Intra4x4 (8.3.1.1; constrained_intra_pred_flag = 0). */
static int i4_neighbour_mode(const gm_encoder *e, int mbx, int mby, int blk, int left)
{
    const gm_mb *cur = &e->mbs[mby * e->mbw + mbx];
    int bx = blk_x[blk], by = blk_y[blk];
    const gm_mb *n = cur;
    int nb;
    if (left) {
        if (bx > 0)
            nb = xy2blk[by][bx - 1];
        else {
            if (mbx == 0)
                return -1;
            n = cur - 1;
            nb = xy2blk[by][3];
        }
    } else {
        if (by > 0)
            nb = xy2blk[by - 1][bx];
        else {
            if (!top_avail(e, mby))
                return -1;
            n = cur - e->mbw;
            nb = xy2blk[3][bx];
        }
    }
    return n->type == GM_MB_I4x4 ? n->i4_mode[nb] : 2;
}

static int i4_pred_mode(const gm_encoder *e, int mbx, int mby, int blk)
{
    int a = i4_neighbour_mode(e, mbx, mby, blk, 1), b = i4_neighbour_mode(e, mbx, mby, blk, 0);
    if (a < 0 || b < 0)
        return 2;
    return a < b ? a : b;
}

/* Tries to code the macroblock's luma as Intra4x4.  Block by block: mode = argmin over available modes of
 * (SAD + lambda * modebits) << 4 | mode with modebits = 1 for the predicted mode, 4 otherwise; the block is
 * reconstructed at once because the next blocks predict from it.  Gives up (returns 0) as soon as the
 * accumulated cost reaches cost16, the cost of the best Intra16x16 mode. */
static int try_intra4x4(gm_encoder *e, int mbx, int mby, uint32_t cost16)
{
    int W = e->W, qp = e->qp, lam = me_lambda(qp);
    gm_mb *mb = &e->mbs[mby * e->mbw + mbx];
    const uint8_t *src = e->src.p[0] + (size_t)(mby * 16) * W + mbx * 16;
    uint8_t *dst = e->unf.p[0] + (size_t)(mby * 16) * W + mbx * 16;
    uint32_t cost4 = 0;
    int cbp = 0;
    mb->type = GM_MB_I4x4; /* i4_pred_mode of later blocks looks at the blocks already decided */
    for (int b = 0; b < 16; b++) {
        int bx = blk_x[b], by = blk_y[b];
        int has_top = by > 0 || top_avail(e, mby), has_left = bx > 0 || mbx > 0;
        int has_tl = (bx > 0 || mbx > 0) && (by > 0 || top_avail(e, mby));
        int has_tr;
        if (by == 0)
            has_tr = top_avail(e, mby) && (bx < 3 || mbx + 1 < e->mbw);
        else
            has_tr = bx < 3 && xy2blk[by - 1][bx + 1] < b;
        const uint8_t *s4 = src + by * 4 * W + bx * 4;
        uint8_t *d4 = dst + by * 4 * W + bx * 4;
        int t[8] = {0}, l[4] = {0}, m = 0;
        if (has_top)
            for (int i = 0; i < 8; i++)
                t[i] = d4[-W + (i < 4 || has_tr ? i : 3)];
        if (has_left)
            for (int i = 0; i < 4; i++)
                l[i] = d4[i * W - 1];
        if (has_tl)
            m = d4[-W - 1];
        int pm = i4_pred_mode(e, mbx, mby, b);
        uint32_t best = 0xffffffffu;
        uint8_t pred[16], bpred[16];
        for (int mode = 0; mode < 9; mode++) {
            int need_top = mode == 0 || mode == 3 || mode == 7 || mode == 4 || mode == 5 || mode == 6;
            int need_left = mode == 1 || mode == 8 || mode == 4 || mode == 5 || mode == 6;
            if ((need_top && !has_top) || (need_left && !has_left) || ((mode >= 4 && mode <= 6) && !has_tl))
                continue;
            pred4x4(mode, t, l, m, has_top, has_left, pred);
            uint32_t cost = (uint32_t)sad_block(s4, W, pred, 4, 4, 4) + (uint32_t)(lam * (mode == pm ? 1 : 4));
            uint32_t key = (cost << 4) | (uint32_t)mode;
            if (key < best) {
                best = key;
                memcpy(bpred, pred, 16);
            }
        }
        cost4 += best >> 4;
        if (cost4 >= cost16)
            return 0;
        mb->i4_mode[b] = (uint8_t)(best & 15);
        int16_t d[16];
        int w[16];
        resid4x4(s4, W, bpred, 4, d);
        fdct4x4(d, w);
        int n = quant_block(w, qp, 1, 0, mb->coef[b]);
        mb->nnz[b] = (uint8_t)n;
        if (n)
            cbp |= 1 << (b >> 2);
        int dq[16] = {0};
        if (n)
            dequant_block(mb->coef[b], qp, 0, dq);
        idct4x4_add(dq, d4, W, bpred, 4);
    }
    /* an 8x8 quadrant without coefficients in any of its blocks is not coded: its cbp bit is 0 already */
    mb->cbp = (uint8_t)cbp;
    return 1;
}

static void encode_mb_intra(gm_encoder *e, int mbx, int mby, int allow_i4)
{
    int W = e->W, CW = W / 2, qp = e->qp;
    gm_mb *mb = &e->mbs[mby * e->mbw + mbx];
    frame_t *out = &e->unf;
    memset(mb, 0, sizeof(*mb));
    mb->type = GM_MB_I16x16;
    int has_top = top_avail(e, mby), has_left = mbx > 0;
    const uint8_t *src = e->src.p[0] + (size_t)(mby * 16) * W + mbx * 16;
    uint8_t *dst = out->p[0] + (size_t)(mby * 16) * W + mbx * 16;

    uint8_t top[16] = {0}, left[16] = {0};
    int tl = 0;
    if (has_top)
        memcpy(top, dst - W, 16);
    if (has_left)
        for (int y = 0; y < 16; y++)
            left[y] = dst[y * W - 1];
    if (has_top && has_left)
        tl = dst[-W - 1];

    /* mode decision: min over available modes of (SAD << 2 | mode) */
    uint8_t pred[256], best_pred[256];
    uint32_t best = 0xffffffffu;
    for (int mode = 0; mode < 4; mode++) {
        if (mode == 0 && !has_top)
            continue;
        if (mode == 1 && !has_left)
            continue;
        if (mode == 3 && !(has_top && has_left))
            continue;
        pred16x16(mode, top, left, tl, has_top, has_left, pred);
        uint32_t key = ((uint32_t)sad_block(src, W, pred, 16, 16, 16) << 2) | (uint32_t)mode;
        if (key < best) {
            best = key;
            memcpy(best_pred, pred, 256);
        }
    }
    mb->i16_mode = (uint8_t)(best & 3);
    int use_i4 = allow_i4 && e->cfg.intra4x4 && try_intra4x4(e, mbx, mby, best >> 2);
    if (use_i4) {
        mb->i16_mode = 0;
    } else {
        memset(mb->coef, 0, sizeof(mb->coef));
        memset(mb->nnz, 0, sizeof(mb->nnz));
        memset(mb->i4_mode, 0, sizeof(mb->i4_mode));
        mb->type = GM_MB_I16x16;

    /* luma: 16 x (transform, AC quant), DC Hadamard + quant */
    int wblk[16][16], dcm[16]; /* dcm raster [by*4+bx] */
    int any_ac = 0;
    for (int b = 0; b < 16; b++) {
        int bx = blk_x[b] * 4, by = blk_y[b] * 4;
        int16_t d[16];
        resid4x4(src + by * W + bx, W, best_pred + by * 16 + bx, 16, d);
        fdct4x4(d, wblk[b]);
        dcm[blk_y[b] * 4 + blk_x[b]] = wblk[b][0];
        int n = quant_block(wblk[b], qp, 1, 1, mb->coef[b]);
        mb->nnz[b] = (uint8_t)n;
        any_ac |= n;
    }
    {
        /* 4x4 Hadamard (unscaled), |Z| = (|Y|*MF0 + 4f) >> (qbits+2) */
        int t[16], yd[16];
        for (int i = 0; i < 4; i++) {
            int a = dcm[i * 4], b = dcm[i * 4 + 1], c = dcm[i * 4 + 2], d = dcm[i * 4 + 3];
            t[i * 4 + 0] = a + b + c + d;
            t[i * 4 + 1] = a + b - c - d;
            t[i * 4 + 2] = a - b - c + d;
            t[i * 4 + 3] = a - b + c - d;
        }
        for (int i = 0; i < 4; i++) {
            int a = t[i], b = t[4 + i], c = t[8 + i], d = t[12 + i];
            yd[i] = a + b + c + d;
            yd[4 + i] = a + b - c - d;
            yd[8 + i] = a - b - c + d;
            yd[12 + i] = a - b + c - d;
        }
        int qbits = 15 + qp / 6, f = (1 << qbits) / 3, n = 0;
        for (int i = 0; i < 16; i++) {
            int z = quant1(yd[h264_zigzag4x4[i]], h264_quant_mf[qp % 6][0], 4 * f, qbits + 2);
            mb->coef[16][i] = (int16_t)z;
            n += z != 0;
        }
        mb->nnz[16] = (uint8_t)n;
    }
    mb->cbp = any_ac ? 15 : 0;
    if (!any_ac)
        for (int b = 0; b < 16; b++)
            mb->nnz[b] = 0;

    /* luma reconstruction */
    {
        int c[16], t[16], fdc[16];
        for (int i = 0; i < 16; i++)
            c[h264_zigzag4x4[i]] = mb->coef[16][i];
        for (int i = 0; i < 4; i++) {
            int a = c[i * 4], b = c[i * 4 + 1], cc = c[i * 4 + 2], d = c[i * 4 + 3];
            t[i * 4 + 0] = a + b + cc + d;
            t[i * 4 + 1] = a + b - cc - d;
            t[i * 4 + 2] = a - b - cc + d;
            t[i * 4 + 3] = a - b + cc - d;
        }
        for (int i = 0; i < 4; i++) {
            int a = t[i], b = t[4 + i], cc = t[8 + i], d = t[12 + i];
            fdc[i] = a + b + cc + d;
            fdc[4 + i] = a + b - cc - d;
            fdc[8 + i] = a - b - cc + d;
            fdc[12 + i] = a - b + cc - d;
        }
        int ls = 16 * h264_dequant_v[qp % 6][0];
        for (int b = 0; b < 16; b++) {
            int bx = blk_x[b] * 4, by = blk_y[b] * 4;
            int d[16] = {0};
            if (any_ac)
                dequant_block(mb->coef[b], qp, 1, d);
            int fv = fdc[blk_y[b] * 4 + blk_x[b]];
            if (qp >= 36)
                d[0] = (fv * ls) * (1 << (qp / 6 - 6));
            else
                d[0] = (fv * ls + (1 << (5 - qp / 6))) >> (6 - qp / 6);
            idct4x4_add(d, dst + by * W + bx, W, best_pred + by * 16 + bx, 16);
        }
    }

    } /* !use_i4 */

    /* chroma */
    uint8_t cpred[2][64], cbest[2][64];
    uint8_t ctop[2][8] = {{0}}, cleft[2][8] = {{0}};
    int ctl[2] = {0, 0};
    for (int c = 0; c < 2; c++) {
        uint8_t *cd = out->p[1 + c] + (size_t)(mby * 8) * CW + mbx * 8;
        if (has_top)
            memcpy(ctop[c], cd - CW, 8);
        if (has_left)
            for (int y = 0; y < 8; y++)
                cleft[c][y] = cd[y * CW - 1];
        if (has_top && has_left)
            ctl[c] = cd[-CW - 1];
    }
    best = 0xffffffffu;
    for (int mode = 0; mode < 4; mode++) {
        if (mode == 1 && !has_left)
            continue;
        if (mode == 2 && !has_top)
            continue;
        if (mode == 3 && !(has_top && has_left))
            continue;
        uint32_t sad = 0;
        for (int c = 0; c < 2; c++) {
            pred_chroma8x8(mode, ctop[c], cleft[c], ctl[c], has_top, has_left, cpred[c]);
            sad += (uint32_t)sad_block(e->src.p[1 + c] + (size_t)(mby * 8) * CW + mbx * 8, CW, cpred[c], 8, 8, 8);
        }
        uint32_t key = (sad << 2) | (uint32_t)mode;
        if (key < best) {
            best = key;
            memcpy(cbest, cpred, sizeof(cbest));
        }
    }
    mb->chroma_mode = (uint8_t)(best & 3);
    encode_chroma(e, mb, mbx, mby, cbest, 1, out);
}

/* ------------------------------------------------------------------------------------------
 * K1 motion estimation: exhaustive integer search, +-R, on the previous deblocked recon with
 * edge-clamped reference fetch.  cost = SAD + lambda * (mvbits(dx) + mvbits(dy)),
 * key = cost << 15 | raster rank; argmin of key (order independent => parallel friendly).
 * ------------------------------------------------------------------------------------------ */
static inline int mv_bits(int d) /* se(v) length of the quarter-pel value 4*d */
{
    if (d == 0)
        return 1;
    int a = iabs(d);
    return 7 + 2 * (31 - __builtin_clz((unsigned)a));
}

static inline int me_lambda(int qp) { return 1 << CLIP3(0, 5, (qp - 12) / 6); }

/* The reference plane is edge-extended once per frame (pad = R + 16) so that the search loops carry no
 * clamping and the compiler can vectorise the SAD; the result is identical to clamped fetches. */
static void pad_reference(gm_encoder *e, const frame_t *ref)
{
    int W = e->W, H = e->H, P = e->cfg.me_range + 16, PW = W + 2 * P;
    if (!e->refpad)
        e->refpad = (uint8_t *)malloc((size_t)PW * (H + 2 * P));
    for (int y = -P; y < H + P; y++) {
        const uint8_t *srow = ref->p[0] + (size_t)CLIP3(0, H - 1, y) * W;
        uint8_t *drow = e->refpad + (size_t)(y + P) * PW;
        memset(drow, srow[0], (size_t)P);
        memcpy(drow + P, srow, (size_t)W);
        memset(drow + P + W, srow[W - 1], (size_t)P);
    }
}

static uint32_t motion_search(gm_encoder *e, const frame_t *ref, int mbx, int mby, int *bdx, int *bdy)
{
    (void)ref;
    int W = e->W, R = e->cfg.me_range, lam = me_lambda(e->qp), P = R + 16, PW = W + 2 * P;
    const uint8_t *src = e->src.p[0] + (size_t)(mby * 16) * W + mbx * 16;
    uint32_t best = 0xffffffffu;
    for (int dy = -R; dy <= R; dy++)
        for (int dx = -R; dx <= R; dx++) {
            const uint8_t *rp = e->refpad + (size_t)(mby * 16 + dy + P) * PW + mbx * 16 + dx + P;
            int sad = 0;
            for (int y = 0; y < 16; y++) {
                const uint8_t *a = src + y * W, *b = rp + (size_t)y * PW;
                for (int x = 0; x < 16; x++)
                    sad += iabs(a[x] - b[x]);
            }
            uint32_t cost = (uint32_t)(sad + lam * (mv_bits(dx) + mv_bits(dy)));
            uint32_t key = (cost << 15) | (uint32_t)((dy + R) * (2 * R + 1) + (dx + R));
            if (key < best) {
                best = key;
                *bdx = dx;
                *bdy = dy;
            }
        }
    return best >> 15; /* cost of the winner */
}

/* p_intra extension (SURVEY 8f rank 2): intra macroblocks inside P frames.  Decision per macroblock, order
 * independent: best Intra16x16 SAD against the neighbours as they are after the ALL-INTER reconstruction of the frame
 * (pass A), chosen when sad16 + 8 * lambda < the motion search's best cost.  The chosen macroblocks are then re-coded
 * as Intra16x16 in raster order with their true neighbours (pass C, encode_mb_intra). */
static int p_intra_decide(gm_encoder *e, int mbx, int mby, uint32_t inter_cost)
{
    int W = e->W, has_top = top_avail(e, mby), has_left = mbx > 0;
    const uint8_t *src = e->src.p[0] + (size_t)(mby * 16) * W + mbx * 16;
    const uint8_t *dst = e->unf.p[0] + (size_t)(mby * 16) * W + mbx * 16;
    uint8_t top[16] = {0}, left[16] = {0}, pred[256];
    int tl = 0;
    if (has_top)
        memcpy(top, dst - W, 16);
    if (has_left)
        for (int y = 0; y < 16; y++)
            left[y] = dst[y * W - 1];
    if (has_top && has_left)
        tl = dst[-W - 1];
    uint32_t best = 0xffffffffu;
    for (int mode = 0; mode < 4; mode++) {
        if ((mode == 0 && !has_top) || (mode == 1 && !has_left) || (mode == 3 && !(has_top && has_left)))
            continue;
        pred16x16(mode, top, left, tl, has_top, has_left, pred);
        uint32_t sad = (uint32_t)sad_block(src, W, pred, 16, 16, 16);
        if (sad < best)
            best = sad;
    }
    return best + 8u * (uint32_t)me_lambda(e->qp) < inter_cost;
}


/* ------------------------------------------------------------------------------------------
 * K3 inter macroblock: integer luma MC, bilinear chroma MC (xFrac,yFrac in {0,4}),
 * transform/quant/dequant/IDCT, reconstruction (before deblocking).
 * ------------------------------------------------------------------------------------------ */
static void encode_mb_inter(gm_encoder *e, const frame_t *ref, int mbx, int mby, int dx, int dy)
{
    int W = e->W, H = e->H, CW = W / 2, CH = H / 2, qp = e->qp;
    gm_mb *mb = &e->mbs[mby * e->mbw + mbx];
    frame_t *out = &e->unf;
    memset(mb, 0, sizeof(*mb));
    mb->type = GM_MB_P16x16;
    mb->mv[0] = (int16_t)(dx * 4);
    mb->mv[1] = (int16_t)(dy * 4);
    const uint8_t *src = e->src.p[0] + (size_t)(mby * 16) * W + mbx * 16;
    uint8_t *dst = out->p[0] + (size_t)(mby * 16) * W + mbx * 16;
    uint8_t pred[256];
    for (int y = 0; y < 16; y++) {
        int ry = CLIP3(0, H - 1, mby * 16 + y + dy);
        for (int x = 0; x < 16; x++)
            pred[y * 16 + x] = ref->p[0][(size_t)ry * W + CLIP3(0, W - 1, mbx * 16 + x + dx)];
    }
    int cbp = 0;
    for (int b = 0; b < 16; b++) {
        int bx = blk_x[b] * 4, by = blk_y[b] * 4, w[16];
        int16_t d[16];
        resid4x4(src + by * W + bx, W, pred + by * 16 + bx, 16, d);
        fdct4x4(d, w);
        int n = quant_block(w, qp, 0, 0, mb->coef[b]);
        mb->nnz[b] = (uint8_t)n;
        if (n)
            cbp |= 1 << (b >> 2);
    }
    mb->cbp = (uint8_t)cbp;
    for (int b = 0; b < 16; b++) {
        int bx = blk_x[b] * 4, by = blk_y[b] * 4;
        int d[16] = {0};
        if (mb->nnz[b])
            dequant_block(mb->coef[b], qp, 0, d);
        idct4x4_add(d, dst + by * W + bx, W, pred + by * 16 + bx, 16);
    }
    /* chroma MC: mvC = luma mv in 1/8 chroma-pel units */
    uint8_t cpred[2][64];
    int mvx = dx * 4, mvy = dy * 4;
    int xi = mvx >> 3, yi = mvy >> 3, xf = mvx & 7, yf = mvy & 7;
    for (int c = 0; c < 2; c++) {
        const uint8_t *rp = ref->p[1 + c];
        for (int y = 0; y < 8; y++) {
            int y0 = CLIP3(0, CH - 1, mby * 8 + y + yi), y1 = CLIP3(0, CH - 1, mby * 8 + y + yi + 1);
            for (int x = 0; x < 8; x++) {
                int x0 = CLIP3(0, CW - 1, mbx * 8 + x + xi), x1 = CLIP3(0, CW - 1, mbx * 8 + x + xi + 1);
                int A = rp[(size_t)y0 * CW + x0], B = rp[(size_t)y0 * CW + x1];
                int C = rp[(size_t)y1 * CW + x0], D = rp[(size_t)y1 * CW + x1];
                cpred[c][y * 8 + x] =
                    (uint8_t)(((8 - xf) * (8 - yf) * A + xf * (8 - yf) * B + (8 - xf) * yf * C + xf * yf * D + 32) >> 6);
            }
        }
    }
    encode_chroma(e, mb, mbx, mby, cpred, 0, out);
}

/* ------------------------------------------------------------------------------------------
 * K2 median MV prediction (16x16 partitions only), P_Skip MV rule, mvd and skip decision.
 * Runs after every MV of the frame is final, so it is order independent.
 * ------------------------------------------------------------------------------------------ */
static inline int median3(int a, int b, int c) { return imax(imin(a, b), imin(imax(a, b), c)); }

static void neighbour_mv(const gm_encoder *e, int mbx, int mby, int avail, int16_t mv[2], int *refidx)
{
    if (!avail) {
        mv[0] = mv[1] = 0;
        *refidx = -1;
        return;
    }
    const gm_mb *n = &e->mbs[mby * e->mbw + mbx];
    if (n->type == GM_MB_P16x16 || n->type == GM_MB_PSKIP) {
        mv[0] = n->mv[0];
        mv[1] = n->mv[1];
        *refidx = 0;
    } else { /* intra */
        mv[0] = mv[1] = 0;
        *refidx = -1;
    }
}

static void predict_mv(const gm_encoder *e, int mbx, int mby, int16_t mvp[2], int16_t skip_mv[2])
{
    int16_t a[2], b[2], c[2];
    int ra, rb, rc;
    int availA = mbx > 0, availB = top_avail(e, mby);
    int availC = availB && mbx + 1 < e->mbw, availD = availB && mbx > 0;
    neighbour_mv(e, mbx - 1, mby, availA, a, &ra);
    neighbour_mv(e, mbx, mby - 1, availB, b, &rb);
    if (availC)
        neighbour_mv(e, mbx + 1, mby - 1, 1, c, &rc);
    else
        neighbour_mv(e, mbx - 1, mby - 1, availD, c, &rc);
    int availCD = availC || availD;
    if (!availB && !availCD && availA) {
        b[0] = c[0] = a[0];
        b[1] = c[1] = a[1];
        rb = rc = ra;
    }
    int match = (ra == 0) + (rb == 0) + (rc == 0);
    if (match == 1) {
        const int16_t *m = ra == 0 ? a : (rb == 0 ? b : c);
        mvp[0] = m[0];
        mvp[1] = m[1];
    } else {
        mvp[0] = (int16_t)median3(a[0], b[0], c[0]);
        mvp[1] = (int16_t)median3(a[1], b[1], c[1]);
    }
    /* P_Skip: uses the ORIGINAL A/B (before the B,C := A substitution) */
    int16_t a0[2], b0[2];
    int ra0, rb0;
    neighbour_mv(e, mbx - 1, mby, availA, a0, &ra0);
    neighbour_mv(e, mbx, mby - 1, availB, b0, &rb0);
    if (!availA || !availB || (ra0 == 0 && a0[0] == 0 && a0[1] == 0) || (rb0 == 0 && b0[0] == 0 && b0[1] == 0)) {
        skip_mv[0] = skip_mv[1] = 0;
    } else {
        skip_mv[0] = mvp[0];
        skip_mv[1] = mvp[1];
    }
}

static void mvp_and_skip(gm_encoder *e)
{
    for (int mby = 0; mby < e->mbh; mby++)
        for (int mbx = 0; mbx < e->mbw; mbx++) {
            gm_mb *mb = &e->mbs[mby * e->mbw + mbx];
            if (mb->type != GM_MB_P16x16)
                continue;
            int16_t mvp[2], smv[2];
            predict_mv(e, mbx, mby, mvp, smv);
            mb->mvd[0] = (int16_t)(mb->mv[0] - mvp[0]);
            mb->mvd[1] = (int16_t)(mb->mv[1] - mvp[1]);
            /* Types are rewritten in place; predict_mv only reads mv[], which never changes,
             * and treats P16x16 and PSKIP alike, so the pass stays order independent. */
            if (mb->cbp == 0 && mb->mv[0] == smv[0] && mb->mv[1] == smv[1]) {
                mb->type = GM_MB_PSKIP;
                mb->mvd[0] = mb->mvd[1] = 0;
            }
        }
}

/* ------------------------------------------------------------------------------------------
 * K5 deblocking filter (H.264 8.7), slice offsets 0 (cedar.c:1024-1029), constant QP.
 * Macroblock raster order; per MB: luma vertical edges, luma horizontal edges, then chroma.
 * ------------------------------------------------------------------------------------------ */
static inline int mb_is_intra(const gm_mb *m) { return m->type == GM_MB_I16x16 || m->type == GM_MB_I4x4; }

/* bS between 4x4 luma block bp of macroblock mp and block bq of mq; mb_edge = on a MB boundary */
static int boundary_strength(const gm_mb *mp, int bp, const gm_mb *mq, int bq, int mb_edge)
{
    if (mb_is_intra(mp) || mb_is_intra(mq))
        return mb_edge ? 4 : 3;
    if (mp->nnz[bp] || mq->nnz[bq])
        return 2;
    if (iabs(mp->mv[0] - mq->mv[0]) >= 4 || iabs(mp->mv[1] - mq->mv[1]) >= 4)
        return 1;
    return 0;
}

/* Filter one line of samples across an edge.  pix points at q0; xs = step across the edge. */
static void filter_line(uint8_t *pix, int xs, int bS, int alpha, int beta, int tc0, int chroma)
{
    int p0 = pix[-1 * xs], p1 = pix[-2 * xs], q0 = pix[0], q1 = pix[1 * xs];
    if (iabs(p0 - q0) >= alpha || iabs(p1 - p0) >= beta || iabs(q1 - q0) >= beta)
        return;
    if (chroma) {
        if (bS < 4) {
            int tc = tc0 + 1;
            int delta = CLIP3(-tc, tc, (((q0 - p0) * 4) + (p1 - q1) + 4) >> 3);
            pix[-xs] = (uint8_t)clip255(p0 + delta);
            pix[0] = (uint8_t)clip255(q0 - delta);
        } else {
            pix[-xs] = (uint8_t)((2 * p1 + p0 + q1 + 2) >> 2);
            pix[0] = (uint8_t)((2 * q1 + q0 + p1 + 2) >> 2);
        }
        return;
    }
    int p2 = pix[-3 * xs], q2 = pix[2 * xs];
    int ap = iabs(p2 - p0), aq = iabs(q2 - q0);
    if (bS < 4) {
        int tc = tc0 + (ap < beta) + (aq < beta);
        int delta = CLIP3(-tc, tc, (((q0 - p0) * 4) + (p1 - q1) + 4) >> 3);
        pix[-xs] = (uint8_t)clip255(p0 + delta);
        pix[0] = (uint8_t)clip255(q0 - delta);
        if (ap < beta)
            pix[-2 * xs] = (uint8_t)(p1 + CLIP3(-tc0, tc0, (p2 + ((p0 + q0 + 1) >> 1) - (p1 << 1)) >> 1));
        if (aq < beta)
            pix[xs] = (uint8_t)(q1 + CLIP3(-tc0, tc0, (q2 + ((p0 + q0 + 1) >> 1) - (q1 << 1)) >> 1));
    } else {
        int p3 = pix[-4 * xs], q3 = pix[3 * xs];
        int strong = iabs(p0 - q0) < ((alpha >> 2) + 2);
        if (ap < beta && strong) {
            pix[-xs] = (uint8_t)((p2 + 2 * p1 + 2 * p0 + 2 * q0 + q1 + 4) >> 3);
            pix[-2 * xs] = (uint8_t)((p2 + p1 + p0 + q0 + 2) >> 2);
            pix[-3 * xs] = (uint8_t)((2 * p3 + 3 * p2 + p1 + p0 + q0 + 4) >> 3);
        } else
            pix[-xs] = (uint8_t)((2 * p1 + p0 + q1 + 2) >> 2);
        if (aq < beta && strong) {
            pix[0] = (uint8_t)((p1 + 2 * p0 + 2 * q0 + 2 * q1 + q2 + 4) >> 3);
            pix[xs] = (uint8_t)((p0 + q0 + q1 + q2 + 2) >> 2);
            pix[2 * xs] = (uint8_t)((2 * q3 + 3 * q2 + q1 + q0 + p0 + 4) >> 3);
        } else
            pix[0] = (uint8_t)((2 * q1 + q0 + p1 + 2) >> 2);
    }
}

static void deblock_mb(gm_encoder *e, frame_t *f, int mbx, int mby)
{
    int W = e->W, CW = W / 2;
    const gm_mb *cur = &e->mbs[mby * e->mbw + mbx];
    int bsv[4][4], bsh[4][4]; /* [edge][segment] */
    for (int edge = 0; edge < 4; edge++)
        for (int s = 0; s < 4; s++) {
            /* vertical edge `edge` at x = 4*edge, segment s covers rows 4s..4s+3 */
            if (edge == 0) {
                if (mbx == 0)
                    bsv[0][s] = 0;
                else
                    bsv[0][s] = boundary_strength(cur - 1, xy2blk[s][3], cur, xy2blk[s][0], 1);
            } else
                bsv[edge][s] = boundary_strength(cur, xy2blk[s][edge - 1], cur, xy2blk[s][edge], 0);
            if (edge == 0) {
                if (mby == 0)
                    bsh[0][s] = 0;
                else
                    bsh[0][s] = boundary_strength(cur - e->mbw, xy2blk[3][s], cur, xy2blk[0][s], 1);
            } else
                bsh[edge][s] = boundary_strength(cur, xy2blk[edge - 1][s], cur, xy2blk[edge][s], 0);
        }
    int qp = e->qp, qpc = e->qpc;
    int alpha = h264_deblock_alpha[qp], beta = h264_deblock_beta[qp];
    int alphac = h264_deblock_alpha[qpc], betac = h264_deblock_beta[qpc];
    uint8_t *y = f->p[0] + (size_t)(mby * 16) * W + mbx * 16;
    for (int edge = 0; edge < 4; edge++) /* luma vertical edges */
        for (int r = 0; r < 16; r++) {
            int bS = bsv[edge][r >> 2];
            if (bS)
                filter_line(y + r * W + edge * 4, 1, bS, alpha, beta, bS < 4 ? h264_deblock_tc0[qp][bS - 1] : 0, 0);
        }
    for (int edge = 0; edge < 4; edge++) /* luma horizontal edges */
        for (int c = 0; c < 16; c++) {
            int bS = bsh[edge][c >> 2];
            if (bS)
                filter_line(y + (edge * 4) * W + c, W, bS, alpha, beta, bS < 4 ? h264_deblock_tc0[qp][bS - 1] : 0, 0);
        }
    for (int pl = 1; pl < 3; pl++) {
        uint8_t *c = f->p[pl] + (size_t)(mby * 8) * CW + mbx * 8;
        for (int edge = 0; edge < 2; edge++) /* chroma vertical edges at x = 0, 4 <-> luma edges 0, 2 */
            for (int r = 0; r < 8; r++) {
                int bS = bsv[edge * 2][r >> 1];
                if (bS)
                    filter_line(c + r * CW + edge * 4, 1, bS, alphac, betac, bS < 4 ? h264_deblock_tc0[qpc][bS - 1] : 0, 1);
            }
        for (int edge = 0; edge < 2; edge++)
            for (int x = 0; x < 8; x++) {
                int bS = bsh[edge * 2][x >> 1];
                if (bS)
                    filter_line(c + (edge * 4) * CW + x, CW, bS, alphac, betac, bS < 4 ? h264_deblock_tc0[qpc][bS - 1] : 0, 1);
            }
    }
}

/* ------------------------------------------------------------------------------------------
 * K6 CAVLC
 * ------------------------------------------------------------------------------------------ */
/* total_coeff of the neighbouring 4x4 block; returns -1 when unavailable.
 * kind 0: luma blkIdx; kind 1/2: Cb/Cr AC block 0..3 */
static int nnz_left(const gm_encoder *e, int mbx, int mby, int kind, int blk)
{
    const gm_mb *cur = &e->mbs[mby * e->mbw + mbx];
    if (kind == 0) {
        int bx = blk_x[blk], by = blk_y[blk];
        if (bx > 0)
            return cur->nnz[xy2blk[by][bx - 1]];
        if (mbx == 0)
            return -1;
        return (cur - 1)->nnz[xy2blk[by][3]];
    }
    int base = 17 + (kind - 1) * 4, bx = blk & 1, by = blk >> 1;
    if (bx > 0)
        return cur->nnz[base + by * 2];
    if (mbx == 0)
        return -1;
    return (cur - 1)->nnz[base + by * 2 + 1];
}

static int nnz_top(const gm_encoder *e, int mbx, int mby, int kind, int blk)
{
    const gm_mb *cur = &e->mbs[mby * e->mbw + mbx];
    if (kind == 0) {
        int bx = blk_x[blk], by = blk_y[blk];
        if (by > 0)
            return cur->nnz[xy2blk[by - 1][bx]];
        if (!top_avail(e, mby))
            return -1;
        return (cur - e->mbw)->nnz[xy2blk[3][bx]];
    }
    int base = 17 + (kind - 1) * 4, bx = blk & 1, by = blk >> 1;
    if (by > 0)
        return cur->nnz[base + bx];
    if (!top_avail(e, mby))
        return -1;
    return (cur - e->mbw)->nnz[base + 2 + bx];
}

static int calc_nc(const gm_encoder *e, int mbx, int mby, int kind, int blk)
{
    int a = nnz_left(e, mbx, mby, kind, blk), b = nnz_top(e, mbx, mby, kind, blk);
    if (a >= 0 && b >= 0)
        return (a + b + 1) >> 1;
    if (a >= 0)
        return a;
    if (b >= 0)
        return b;
    return 0;
}

/* residual_block_cavlc: lev = zig-zag levels [first .. first+max-1]; nC < 0 => chroma DC */
static void cavlc_block(bitw *bw, const int16_t *lev, int max_coeff, int nC)
{
    int16_t lv[16];
    int run[16];
    int total = 0, zeros = 0, last = -1;
    /* gather non-zero coefficients in reverse scan order */
    for (int i = max_coeff - 1; i >= 0; i--)
        if (lev[i]) {
            if (last < 0) {
                last = i;
            }
            lv[total] = lev[i];
            int r = 0;
            for (int j = i - 1; j >= 0 && !lev[j]; j--)
                r++;
            run[total] = r;
            total++;
        }
    if (total)
        zeros = last + 1 - total;
    int t1 = 0;
    while (t1 < 3 && t1 < total && iabs(lv[t1]) == 1)
        t1++;
    /* coeff_token */
    if (nC < 0)
        bw_put(bw, h264_chroma_dc_coeff_token_bits[4 * total + t1], h264_chroma_dc_coeff_token_len[4 * total + t1]);
    else {
        int tab = nC < 2 ? 0 : (nC < 4 ? 1 : (nC < 8 ? 2 : 3));
        bw_put(bw, h264_coeff_token_bits[tab][4 * total + t1], h264_coeff_token_len[tab][4 * total + t1]);
    }
    if (!total)
        return;
    for (int i = 0; i < t1; i++)
        bw_put(bw, lv[i] < 0, 1);
    int suffix_len = (total > 10 && t1 < 3) ? 1 : 0;
    for (int i = t1; i < total; i++) {
        int level = lv[i];
        int code = level > 0 ? 2 * level - 2 : -2 * level - 1;
        if (i == t1 && t1 < 3)
            code -= 2;
        if (suffix_len == 0) {
            if (code < 14)
                bw_put(bw, 1, code + 1);
            else if (code < 30) {
                bw_put(bw, 1, 15);
                bw_put(bw, (uint32_t)(code - 14), 4);
            } else {
                /* escape: level_prefix >= 15 */
                int c = code - 30, prefix = 15;
                while (c >= (1 << (prefix - 3))) {
                    c -= 1 << (prefix - 3);
                    prefix++;
                }
                bw_put(bw, 1, prefix + 1);
                bw_put(bw, (uint32_t)c, prefix - 3);
            }
        } else {
            if (code < (15 << suffix_len)) {
                bw_put(bw, 1, (code >> suffix_len) + 1);
                bw_put(bw, (uint32_t)(code & ((1 << suffix_len) - 1)), suffix_len);
            } else {
                int c = code - (15 << suffix_len), prefix = 15;
                while (c >= (1 << (prefix - 3))) {
                    c -= 1 << (prefix - 3);
                    prefix++;
                }
                bw_put(bw, 1, prefix + 1);
                bw_put(bw, (uint32_t)c, prefix - 3);
            }
        }
        if (suffix_len == 0)
            suffix_len = 1;
        if (iabs(level) > (3 << (suffix_len - 1)) && suffix_len < 6)
            suffix_len++;
    }
    if (total < max_coeff) {
        if (nC < 0)
            bw_put(bw, h264_chroma_dc_total_zeros_bits[total - 1][zeros], h264_chroma_dc_total_zeros_len[total - 1][zeros]);
        else
            bw_put(bw, h264_total_zeros_bits[total - 1][zeros], h264_total_zeros_len[total - 1][zeros]);
    }
    int zeros_left = zeros;
    for (int i = 0; i < total - 1 && zeros_left > 0; i++) {
        int zl = imin(zeros_left, 7) - 1;
        bw_put(bw, h264_run_before_bits[zl][run[i]], h264_run_before_len[zl][run[i]]);
        zeros_left -= run[i];
    }
}

static void cavlc_residual(gm_encoder *e, bitw *bw, int mbx, int mby)
{
    const gm_mb *mb = &e->mbs[mby * e->mbw + mbx];
    int cbpl = mb->cbp & 15, cbpc = mb->cbp >> 4;
    if (mb->type == GM_MB_I16x16) {
        cavlc_block(bw, mb->coef[16], 16, calc_nc(e, mbx, mby, 0, 0));
        if (cbpl)
            for (int b = 0; b < 16; b++)
                cavlc_block(bw, mb->coef[b] + 1, 15, calc_nc(e, mbx, mby, 0, b));
    } else {
        for (int b = 0; b < 16; b++)
            if (cbpl & (1 << (b >> 2)))
                cavlc_block(bw, mb->coef[b], 16, calc_nc(e, mbx, mby, 0, b));
    }
    if (cbpc) {
        cavlc_block(bw, mb->coef[17], 4, -1);
        cavlc_block(bw, mb->coef[17] + 4, 4, -1);
    }
    if (cbpc == 2)
        for (int c = 0; c < 2; c++)
            for (int b = 0; b < 4; b++)
                cavlc_block(bw, mb->coef[18 + c * 4 + b] + 1, 15, calc_nc(e, mbx, mby, 1 + c, b));
}

static void cavlc_slice_data(gm_encoder *e, bitw *bw, int frame_i, int row0, int row1)
{
    int skip_run = 0;
    for (int mby = row0; mby < row1; mby++)
        for (int mbx = 0; mbx < e->mbw; mbx++) {
            const gm_mb *mb = &e->mbs[mby * e->mbw + mbx];
            if (mb->type == GM_MB_PSKIP) {
                skip_run++;
                continue;
            }
            if (!frame_i) {
                bw_ue(bw, (uint32_t)skip_run);
                skip_run = 0;
            }
            if (mb->type == GM_MB_I16x16) {
                int t = 1 + mb->i16_mode + 4 * (mb->cbp >> 4) + ((mb->cbp & 15) ? 12 : 0);
                bw_ue(bw, (uint32_t)(t + (frame_i ? 0 : 5)));
                bw_ue(bw, mb->chroma_mode);
                bw_se(bw, 0); /* mb_qp_delta */
            } else if (mb->type == GM_MB_I4x4) {
                bw_ue(bw, frame_i ? 0 : 5); /* I_NxN */
                for (int b = 0; b < 16; b++) {
                    int pm = i4_pred_mode(e, mbx, mby, b), mode = mb->i4_mode[b];
                    if (mode == pm)
                        bw_put(bw, 1, 1); /* prev_intra4x4_pred_mode_flag */
                    else {
                        bw_put(bw, 0, 1);
                        bw_put(bw, (uint32_t)(mode < pm ? mode : mode - 1), 3); /* rem_intra4x4_pred_mode */
                    }
                }
                bw_ue(bw, mb->chroma_mode);
                bw_ue(bw, h264_cbp_to_codenum_intra[mb->cbp]);
                if (mb->cbp)
                    bw_se(bw, 0); /* mb_qp_delta */
            } else {          /* P_L0_16x16 */
                bw_ue(bw, 0);
                bw_se(bw, mb->mvd[0]);
                bw_se(bw, mb->mvd[1]);
                bw_ue(bw, h264_cbp_to_codenum_inter[mb->cbp]);
                if (mb->cbp)
                    bw_se(bw, 0); /* mb_qp_delta */
            }
            cavlc_residual(e, bw, mbx, mby);
        }
    if (skip_run)
        bw_ue(bw, (uint32_t)skip_run);
    /* rbsp_slice_trailing_bits */
    bw_put(bw, 1, 1);
    while (bw->nbits & 7)
        bw_put(bw, 0, 1);
}

/* ------------------------------------------------------------------------------------------
 * K7 CABAC (H.264 9.3): spec-literal arithmetic encoder (9.3.4) and binarisations.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    bitw *bw;
    uint32_t low, range;
    int first_bit, outstanding;
    uint8_t state[1024]; /* pStateIdx << 1 | valMPS */
    int run_max, run_carry; /* longest run of outstanding bits, and the bit that ended it (1 = a carry) */
} cabac_t;

static void cabac_init(cabac_t *c, bitw *bw, int frame_i, int qp)
{
    c->bw = bw;
    c->low = 0;
    c->range = 510;
    c->first_bit = 1;
    c->outstanding = 0;
    c->run_max = 0;
    c->run_carry = 0;
    for (int i = 0; i < 460; i++) {
        int m = frame_i ? h264_cabac_init_I[i][0] : h264_cabac_init_P0[i][0];
        int n = frame_i ? h264_cabac_init_I[i][1] : h264_cabac_init_P0[i][1];
        int pre = CLIP3(1, 126, ((m * CLIP3(0, 51, qp)) >> 4) + n);
        if (pre <= 63)
            c->state[i] = (uint8_t)((63 - pre) << 1);
        else
            c->state[i] = (uint8_t)(((pre - 64) << 1) | 1);
    }
}

static void cabac_put_bit(cabac_t *c, int b)
{
    if (c->outstanding > c->run_max) {
        c->run_max = c->outstanding;
        c->run_carry = b;
    }
    if (c->first_bit)
        c->first_bit = 0;
    else
        bw_put(c->bw, (uint32_t)b, 1);
    while (c->outstanding > 0) {
        bw_put(c->bw, (uint32_t)(1 - b), 1);
        c->outstanding--;
    }
}

static void cabac_renorm(cabac_t *c)
{
    while (c->range < 256) {
        if (c->low < 256)
            cabac_put_bit(c, 0);
        else if (c->low >= 512) {
            c->low -= 512;
            cabac_put_bit(c, 1);
        } else {
            c->low -= 256;
            c->outstanding++;
        }
        c->range <<= 1;
        c->low <<= 1;
    }
}

static void cabac_decision(cabac_t *c, int ctx, int bin)
{
    int st = c->state[ctx] >> 1, mps = c->state[ctx] & 1;
    uint32_t lps = h264_range_lps[st][(c->range >> 6) & 3];
    c->range -= lps;
    if (bin != mps) {
        c->low += c->range;
        c->range = lps;
        if (st == 0)
            mps = 1 - mps;
        st = h264_next_state_lps[st];
    } else
        st = h264_next_state_mps[st];
    c->state[ctx] = (uint8_t)((st << 1) | mps);
    cabac_renorm(c);
}

static void cabac_bypass(cabac_t *c, int bin)
{
    c->low <<= 1;
    if (bin)
        c->low += c->range;
    if (c->low >= 1024) {
        cabac_put_bit(c, 1);
        c->low -= 1024;
    } else if (c->low < 512)
        cabac_put_bit(c, 0);
    else {
        c->low -= 512;
        c->outstanding++;
    }
}

static void cabac_terminate(cabac_t *c, int bin)
{
    c->range -= 2;
    if (bin) {
        c->low += c->range;
        c->range = 2;
        cabac_renorm(c);
        cabac_put_bit(c, (c->low >> 9) & 1);
        bw_put(c->bw, ((c->low >> 7) & 3) | 1, 2); /* includes rbsp_stop_one_bit */
    } else
        cabac_renorm(c);
}

static void cabac_ueg_bypass(cabac_t *c, int k, int v) /* Exp-Golomb order k suffix */
{
    while (v >= (1 << k)) {
        cabac_bypass(c, 1);
        v -= 1 << k;
        k++;
    }
    cabac_bypass(c, 0);
    while (k--)
        cabac_bypass(c, (v >> k) & 1);
}

static const int cat_cbf_off[5] = {0, 4, 8, 12, 16};
static const int cat_sig_off[5] = {0, 15, 29, 44, 47};
static const int cat_abs_off[5] = {0, 10, 20, 30, 39};

/* coded_block_flag of the neighbouring block for ctxIdxInc; `intra` = current MB is intra.
 * cat 0: I16 DC; 1/2: luma block blk; 3: chroma DC of plane comp; 4: chroma AC block blk of comp */
static int cbf_neighbour(const gm_encoder *e, int mbx, int mby, int cat, int comp, int blk, int left, int intra)
{
    const gm_mb *cur = &e->mbs[mby * e->mbw + mbx];
    const gm_mb *n = left ? cur - 1 : cur - e->mbw;
    int navail = left ? mbx > 0 : top_avail(e, mby);
    if (cat == 0) {
        if (!navail)
            return intra;
        return n->type == GM_MB_I16x16 ? n->nnz[16] != 0 : 0;
    }
    if (cat == 3) {
        if (!navail)
            return intra;
        return n->nnz[25 + comp] != 0;
    }
    int v = left ? nnz_left(e, mbx, mby, cat == 4 ? 1 + comp : 0, blk) : nnz_top(e, mbx, mby, cat == 4 ? 1 + comp : 0, blk);
    if (v < 0)
        return intra;
    return v != 0;
}

/* residual_block_cabac for levels lev[0..n-1] (zig-zag order) */
static void cabac_block(cabac_t *c, const int16_t *lev, int n, int cat, int cbf_inc)
{
    int last = -1;
    for (int i = 0; i < n; i++)
        if (lev[i])
            last = i;
    cabac_decision(c, 85 + cat_cbf_off[cat] + cbf_inc, last >= 0);
    if (last < 0)
        return;
    for (int i = 0; i < n - 1; i++) {
        int inc = cat == 3 ? imin(i, 2) : i;
        if (lev[i]) {
            cabac_decision(c, 105 + cat_sig_off[cat] + inc, 1);
            cabac_decision(c, 166 + cat_sig_off[cat] + inc, i == last);
            if (i == last)
                break;
        } else
            cabac_decision(c, 105 + cat_sig_off[cat] + inc, 0);
    }
    int eq1 = 0, gt1 = 0;
    for (int i = last; i >= 0; i--) {
        if (!lev[i])
            continue;
        int a = iabs(lev[i]) - 1;
        int ctx = 227 + cat_abs_off[cat] + (gt1 ? 0 : imin(4, 1 + eq1));
        if (a == 0) {
            cabac_decision(c, ctx, 0);
            eq1++;
        } else {
            cabac_decision(c, ctx, 1);
            ctx = 227 + cat_abs_off[cat] + 5 + imin(4 - (cat == 3), gt1);
            int pre = imin(a, 14);
            for (int j = 1; j < pre; j++)
                cabac_decision(c, ctx, 1);
            if (a < 14)
                cabac_decision(c, ctx, 0);
            else
                cabac_ueg_bypass(c, 0, a - 14);
            gt1++;
        }
        cabac_bypass(c, lev[i] < 0);
    }
}

static void cabac_mvd(cabac_t *c, int base, int mvd, int sum_abs)
{
    int inc = sum_abs < 3 ? 0 : (sum_abs > 32 ? 2 : 1);
    static const int ctxes[8] = {3, 4, 5, 6, 6, 6, 6, 6};
    int a = iabs(mvd);
    if (a == 0) {
        cabac_decision(c, base + inc, 0);
        return;
    }
    cabac_decision(c, base + inc, 1);
    int pre = imin(a, 9);
    for (int i = 1; i < pre; i++)
        cabac_decision(c, base + ctxes[i - 1], 1);
    if (a < 9)
        cabac_decision(c, base + ctxes[pre - 1], 0);
    else
        cabac_ueg_bypass(c, 3, a - 9);
    cabac_bypass(c, mvd < 0);
}

static void cabac_mb(gm_encoder *e, cabac_t *c, int mbx, int mby, int frame_i)
{
    const gm_mb *mb = &e->mbs[mby * e->mbw + mbx];
    const gm_mb *A = mbx > 0 ? mb - 1 : NULL, *B = top_avail(e, mby) ? mb - e->mbw : NULL;
    int intra = mb_is_intra(mb);
    if (!frame_i) {
        int inc = (A && A->type != GM_MB_PSKIP) + (B && B->type != GM_MB_PSKIP);
        cabac_decision(c, 11 + inc, mb->type == GM_MB_PSKIP);
        if (mb->type == GM_MB_PSKIP)
            return;
    }
    int cbpl = mb->cbp & 15, cbpc = mb->cbp >> 4;
    if (mb->type == GM_MB_I16x16) {
        int c0, c1, c2, c3, c4, c5;
        if (frame_i) {
            int inc = (A && A->type != GM_MB_I4x4) + (B && B->type != GM_MB_I4x4);
            c0 = 3 + inc, c1 = 3 + 3, c2 = 3 + 4, c3 = 3 + 5, c4 = 3 + 6, c5 = 3 + 7;
        } else {
            cabac_decision(c, 14, 1); /* prefix: intra in P slice */
            c0 = 17, c1 = 17 + 1, c2 = 17 + 2, c3 = 17 + 2, c4 = 17 + 3, c5 = 17 + 3;
        }
        cabac_decision(c, c0, 1);
        cabac_terminate(c, 0);
        cabac_decision(c, c1, cbpl != 0);
        if (cbpc == 0)
            cabac_decision(c, c2, 0);
        else {
            cabac_decision(c, c2, 1);
            cabac_decision(c, c3, cbpc >> 1);
        }
        cabac_decision(c, c4, mb->i16_mode >> 1);
        cabac_decision(c, c5, mb->i16_mode & 1);
    } else if (mb->type == GM_MB_I4x4) {
        if (frame_i) {
            int inc = (A && A->type != GM_MB_I4x4) + (B && B->type != GM_MB_I4x4);
            cabac_decision(c, 3 + inc, 0); /* I_NxN */
        } else {
            cabac_decision(c, 14, 1);
            cabac_decision(c, 17, 0);
        }
        for (int b = 0; b < 16; b++) {
            int pm = i4_pred_mode(e, mbx, mby, b), mode = mb->i4_mode[b];
            cabac_decision(c, 68, mode == pm);
            if (mode != pm) {
                int rem = mode < pm ? mode : mode - 1;
                cabac_decision(c, 69, rem & 1);
                cabac_decision(c, 69, (rem >> 1) & 1);
                cabac_decision(c, 69, (rem >> 2) & 1);
            }
        }
    } else { /* P_L0_16x16 */
        cabac_decision(c, 14, 0);
        cabac_decision(c, 15, 0);
        cabac_decision(c, 16, 0);
    }
    if (intra) {
        int inc = (A && mb_is_intra(A) && A->chroma_mode != 0) + (B && mb_is_intra(B) && B->chroma_mode != 0);
        int m = mb->chroma_mode;
        cabac_decision(c, 64 + inc, m > 0);
        if (m > 0) {
            cabac_decision(c, 64 + 3, m > 1);
            if (m > 1)
                cabac_decision(c, 64 + 3, m > 2);
        }
    } else {
        for (int k = 0; k < 2; k++) {
            int sa = (A && A->type == GM_MB_P16x16 ? iabs(A->mvd[k]) : 0) +
                     (B && B->type == GM_MB_P16x16 ? iabs(B->mvd[k]) : 0);
            cabac_mvd(c, k ? 47 : 40, mb->mvd[k], sa);
        }
    }
    if (mb->type != GM_MB_I16x16) {
        /* coded_block_pattern: luma (one bin per 8x8), then chroma */
        int cbp_a = A ? (A->cbp & 15) : 15, cbp_b = B ? (B->cbp & 15) : 15; /* unavailable => condTerm 0 */
        for (int b8 = 0; b8 < 4; b8++) {
            int la, lb; /* is the neighbouring 8x8's cbp bit set? */
            if (b8 & 1)
                la = (cbpl >> (b8 - 1)) & 1;
            else
                la = (cbp_a >> (b8 + 1)) & 1;
            if (b8 & 2)
                lb = (cbpl >> (b8 - 2)) & 1;
            else
                lb = (cbp_b >> (b8 + 2)) & 1;
            cabac_decision(c, 73 + (!la) + 2 * (!lb), (cbpl >> b8) & 1);
        }
        int ca = A ? (A->cbp >> 4) : 0, cb = B ? (B->cbp >> 4) : 0;
        cabac_decision(c, 77 + (ca > 0) + 2 * (cb > 0), cbpc > 0);
        if (cbpc > 0)
            cabac_decision(c, 77 + 4 + (ca == 2) + 2 * (cb == 2), cbpc == 2);
    }
    if (mb->type == GM_MB_I16x16 || mb->cbp)
        cabac_decision(c, 60, 0); /* mb_qp_delta = 0; previous delta is always 0 => ctxIdxInc 0 */
    /* residual */
    if (mb->type == GM_MB_I16x16) {
        int inc = cbf_neighbour(e, mbx, mby, 0, 0, 0, 1, intra) + 2 * cbf_neighbour(e, mbx, mby, 0, 0, 0, 0, intra);
        cabac_block(c, mb->coef[16], 16, 0, inc);
        if (cbpl)
            for (int b = 0; b < 16; b++) {
                inc = cbf_neighbour(e, mbx, mby, 1, 0, b, 1, intra) + 2 * cbf_neighbour(e, mbx, mby, 1, 0, b, 0, intra);
                cabac_block(c, mb->coef[b] + 1, 15, 1, inc);
            }
    } else {
        for (int b = 0; b < 16; b++)
            if (cbpl & (1 << (b >> 2))) {
                int inc = cbf_neighbour(e, mbx, mby, 2, 0, b, 1, intra) + 2 * cbf_neighbour(e, mbx, mby, 2, 0, b, 0, intra);
                cabac_block(c, mb->coef[b], 16, 2, inc);
            }
    }
    if (cbpc) {
        for (int comp = 0; comp < 2; comp++) {
            int inc = cbf_neighbour(e, mbx, mby, 3, comp, 0, 1, intra) + 2 * cbf_neighbour(e, mbx, mby, 3, comp, 0, 0, intra);
            cabac_block(c, mb->coef[17] + comp * 4, 4, 3, inc);
        }
    }
    if (cbpc == 2)
        for (int comp = 0; comp < 2; comp++)
            for (int b = 0; b < 4; b++) {
                int inc = cbf_neighbour(e, mbx, mby, 4, comp, b, 1, intra) + 2 * cbf_neighbour(e, mbx, mby, 4, comp, b, 0, intra);
                cabac_block(c, mb->coef[18 + comp * 4 + b] + 1, 15, 4, inc);
            }
}

static void cabac_slice_data(gm_encoder *e, bitw *bw, int frame_i, int row0, int row1)
{
    while (bw->nbits & 7)
        bw_put(bw, 1, 1); /* cabac_alignment_one_bit */
    cabac_t c;
    cabac_init(&c, bw, frame_i, e->qp);
    int n = e->mbw * row1;
    for (int i = e->mbw * row0; i < n; i++) {
        cabac_mb(e, &c, i % e->mbw, i / e->mbw, frame_i);
        cabac_terminate(&c, i == n - 1); /* end_of_slice_flag */
    }
    while (bw->nbits & 7)
        bw_put(bw, 0, 1); /* rbsp_alignment_zero_bit */
}

/* One slice's RBSP from raw bins in the product's bin format (16 bits: ctxIdx in bits 0..9, 1 << 10 bypass,
 * 1 << 11 terminate, value in bit 15): header bits, cabac_alignment_one_bits, the bins through the coder above, and
 * the stop bit and zero padding of the final terminate(1), which must be the last bin and the only terminate(1). */
int gm_cabac_code_bins(const uint16_t *bins, int n, int frame_i, int qp, uint64_t hdr_bits, int hdr_nbits, uint8_t *out,
                       int cap, uint8_t *pre, int *stats)
{
    if (n < 1 || hdr_nbits < 0 || hdr_nbits > 64 || bins[n - 1] != (1u << 11 | 1u << 15))
        return -EINVAL;
    for (int i = 0; i < n; i++)
        if ((bins[i] & 0x7000) || (bins[i] & 0x0c00) == 0x0c00 || (!(bins[i] & 0x0c00) && (bins[i] & 0x3ff) >= 460) ||
            (i + 1 < n && bins[i] == (1u << 11 | 1u << 15)))
            return -EINVAL;
    bitw bw;
    bw_init(&bw, out, (size_t)cap);
    if (hdr_nbits > 32)
        bw_put(&bw, (uint32_t)(hdr_bits >> 32), hdr_nbits - 32);
    bw_put(&bw, (uint32_t)hdr_bits, hdr_nbits > 32 ? 32 : hdr_nbits);
    while (bw.nbits & 7)
        bw_put(&bw, 1, 1); /* cabac_alignment_one_bit */
    const size_t data0 = bw.nbits;
    cabac_t c;
    cabac_init(&c, &bw, frame_i, qp);
    for (int i = 0; i < n; i++) {
        const int v = bins[i] >> 15;
        if (bins[i] & (1u << 11))
            cabac_terminate(&c, v);
        else if (bins[i] & (1u << 10))
            cabac_bypass(&c, v);
        else {
            if (pre)
                pre[i] = c.state[bins[i] & 0x3ff];
            cabac_decision(&c, bins[i] & 0x3ff, v);
        }
    }
    if (stats) {
        stats[0] = c.run_max;
        stats[1] = c.run_carry;
        stats[2] = (int)(bw.nbits - data0); /* slice data bits up to and including the stop bit */
    }
    while (bw.nbits & 7)
        bw_put(&bw, 0, 1);
    if ((bw.nbits >> 3) >= (size_t)cap) /* bw_put stops at cap */
        return -ENOMEM;
    return (int)(bw.nbits >> 3);
}

/* ------------------------------------------------------------------------------------------
 * Per-frame control flow: restates cedar_slashdev_ioctl_encode (cedar.c:1032-1209) with the
 * hardware trigger (:1176) replaced by the macroblock pipeline above.
 * ------------------------------------------------------------------------------------------ */
int gm_encode_frame(gm_encoder *e, const uint8_t *luma, const uint8_t *chroma, uint8_t *out, int out_cap)
{
    int frame_i = e->frame_p_count == 0; /* cedar.c:1047-1050 */
    int n = 0, r;
    ingest(e, luma, chroma);

    if (!e->frame_count || (e->cfg.repeat_headers && frame_i)) { /* cedar.c:1058-1061: once; extension: every IDR */
        if ((r = gm_write_sps(&e->cfg, out + n, out_cap - n)) < 0)
            return r;
        n += r;
        if ((r = gm_write_pps(&e->cfg, out + n, out_cap - n)) < 0)
            return r;
        n += r;
    }

    frame_t *cur = &e->rec[e->cur], *ref = &e->rec[e->cur ^ 1];
    if (frame_i) {
        for (int mby = 0; mby < e->mbh; mby++)
            for (int mbx = 0; mbx < e->mbw; mbx++)
                encode_mb_intra(e, mbx, mby, 1);
    } else {
        pad_reference(e, ref);
        for (int mby = 0; mby < e->mbh; mby++)
            for (int mbx = 0; mbx < e->mbw; mbx++) {
                int dx = 0, dy = 0;
                uint32_t cost = motion_search(e, ref, mbx, mby, &dx, &dy);
                encode_mb_inter(e, ref, mbx, mby, dx, dy);
                if (e->cfg.p_intra)
                    e->inter_cost[mby * e->mbw + mbx] = cost;
            }
        if (e->cfg.p_intra) {
            for (int i = 0; i < e->mbw * e->mbh; i++)
                e->want_intra[i] = (uint8_t)p_intra_decide(e, i % e->mbw, i / e->mbw, e->inter_cost[i]);
            for (int i = 0; i < e->mbw * e->mbh; i++)
                if (e->want_intra[i])
                    encode_mb_intra(e, i % e->mbw, i / e->mbw, 0);
        }
        mvp_and_skip(e);
    }
    for (int p = 0; p < 3; p++)
        memcpy(cur->p[p], e->unf.p[p], (size_t)e->W * e->H / (p ? 4 : 1));
    for (int mby = 0; mby < e->mbh; mby++)
        for (int mbx = 0; mbx < e->mbw; mbx++)
            deblock_mb(e, cur, mbx, mby);

    /* slice NALs: header bits (cedar.c:1063-1066), then slice data.  One slice per picture as in the
     * reference (cedar.c:992-993) unless the slice_rows extension splits the picture into slices of whole
     * macroblock rows. */
    int cabac = e->cfg.entropy_coding_mode == GM_ENTROPY_CABAC;
    for (int row0 = 0; row0 < e->mbh; row0 += e->srows) {
        int row1 = imin(row0 + e->srows, e->mbh);
        bitw bw;
        bw_init(&bw, e->rbsp, e->rbsp_cap);
        write_slice_header(&bw, frame_i, e->frame_p_count, cabac, row0 * e->mbw);
        if (cabac)
            cabac_slice_data(e, &bw, frame_i, row0, row1);
        else
            cavlc_slice_data(e, &bw, frame_i, row0, row1);
        if ((bw.nbits >> 3) >= e->rbsp_cap)
            return -ENOMEM;
        if (out_cap - n < 5)
            return -ENOMEM;
        n += (int)put_startcode(out + n, frame_i ? 3 : 2, frame_i ? 5 : 1);
        size_t esc = epb_copy(out + n, (size_t)(out_cap - n), e->rbsp, bw.nbits >> 3);
        if (esc > (size_t)(out_cap - n))
            return -ENOMEM;
        n += (int)esc;
    }

    double sse = 0;
    for (size_t i = 0; i < (size_t)e->W * e->H; i++) {
        int d = cur->p[0][i] - e->src.p[0][i];
        sse += d * d;
    }
    e->last_sse_y = sse;
    e->last_frame_i = frame_i;

    /* cedar.c:1193-1201 */
    e->frame_p_count++;
    if (e->frame_p_count == e->cfg.keyframe_interval)
        e->frame_p_count = 0;
    e->frame_count++;
    e->cur ^= 1;
    return n;
}
