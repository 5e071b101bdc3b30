/*
 * ORACLE -- TEST INFRASTRUCTURE ONLY.
 *
 * Single-threaded CPU golden model of the CQP I+P H.264 encoder whose CUDA implementation
 * lives in cedarx_h264_encoder_b200/csrc/.  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may build, link or call this code.
 *
 * What is pinned by the reference and what is not:
 *   - Stream framing, SPS, PPS, slice headers, GOP/frame counters, what is emitted when, and the configuration rules
 *     restate /root/reference/kernel/cedar.c:187-223 (bit writer, Exp-Golomb), :868-890 (start code, trailing-bits
 *     quirk), :892-937 (SPS), :939-982 (PPS), :984-1030 (slice header), :1047-1066 (what is emitted when), :1193-1201
 *     (GOP counter, reference swap), :744-832 / userspace/h264enc.c:50-66,178-187 (configuration).  PINNED BY THE
 *     REFERENCE ITSELF, EXECUTED: oracle/refsim compiles kernel/cedar.c and userspace/h264enc.c unmodified (from where
 *     they lie) against a software model of the video engine's registers; this model's streams equal what that driver
 *     returns frame by frame (tests/test_refsim.py), and tests/golden/headers.json + ref_streams.json are generated
 *     from it (tests/golden/make_ref_headers.py).
 *   - Slice data (everything per macroblock): the reference has NO source for it -- it is Allwinner A20 silicon
 *     started by kernel/cedar.c:1176 (in refsim this model IS the engine behind that trigger).  PARITY UNPINNED by
 *     the reference; pinned instead by (a) an independent conformant decoder (libavcodec) reproducing this model's
 *     reconstruction bit-exactly and (b) committed golden bitstream hashes.
 */
#ifndef H264_GOLDEN_H
#define H264_GOLDEN_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GM_FORMAT_NV12 0 /* kernel/cedar_ioctl.h:15 */
#define GM_FORMAT_NV16 1 /* kernel/cedar_ioctl.h:16 */
#define GM_ENTROPY_CAVLC 0 /* kernel/cedar_ioctl.h:30 */
#define GM_ENTROPY_CABAC 1 /* kernel/cedar_ioctl.h:31 */

#define GM_MB_I16x16 0
#define GM_MB_P16x16 1
#define GM_MB_PSKIP 2
#define GM_MB_I4x4 3

/* Same field names as struct cedar_ioctl_config (kernel/cedar_ioctl.h:12-32) + extensions. */
typedef struct gm_config {
    int src_width, src_height, src_format;
    int dst_width, dst_height;
    int profile, level, qp, keyframe_interval;
    int entropy_coding_mode;
    int me_range;      /* extension: integer-pel full-search radius (default 16) */
    int relax_gop;     /* extension: accept keyframe_interval >= 32 (cedar.c:784-789 rejects) */
    int intra4x4;      /* extension: enable Intra4x4 macroblocks in I frames */
    int slice_rows;    /* extension: macroblock rows per slice; 0 = one slice per picture (cedar.c:992-993) */
    int sps_crop;      /* extension: frame cropping to src_width x src_height in the SPS (dead in the reference) */
    int auto_level;    /* extension: level_idc from the picture size instead of cfg->level */
    int repeat_headers; /* extension: SPS + PPS before every IDR picture (cedar.c:1058-1061 writes them once) */
    int p_intra;       /* extension: Intra16x16 macroblocks inside P frames where they beat the motion search */
} gm_config;

/* Per-macroblock record: every syntax element the entropy coder needs. */
typedef struct gm_mb {
    uint8_t type;        /* GM_MB_* */
    uint8_t i16_mode;    /* Intra16x16PredMode: 0 V, 1 H, 2 DC, 3 Plane */
    uint8_t chroma_mode; /* intra_chroma_pred_mode: 0 DC, 1 H, 2 V, 3 Plane */
    uint8_t cbp;         /* luma 4 bits | chroma (0..2) << 4 */
    int16_t mv[2];       /* quarter-pel, always multiples of 4 */
    int16_t mvd[2];      /* mv - median prediction */
    /* total_coeff per block: 0..15 luma (luma4x4BlkIdx order; AC count for I16x16),
     * 16 Intra16x16 DC, 17..20 Cb AC, 21..24 Cr AC, 25 Cb DC, 26 Cr DC */
    uint8_t nnz[27];
    uint8_t i4_mode[16]; /* Intra4x4PredMode per luma4x4BlkIdx */
    /* levels in zig-zag order: blocks 0..15 luma, 16 I16 DC, 17 chroma DC (Cb 0..3, Cr 4..7),
     * 18..21 Cb AC, 22..25 Cr AC (index 0 unused for AC blocks) */
    int16_t coef[26][16];
} gm_mb;

typedef struct gm_encoder gm_encoder;

/* Returns 0 or a negative errno exactly as cedar_slashdev_ioctl_config would (cedar.c:744-789). */
int gm_open(const gm_config *cfg, gm_encoder **out);
/* luma: src_width*src_height bytes; chroma: interleaved CbCr, src_width*src_height/2 (NV12) or
 * src_width*src_height (NV16) bytes (userspace/h264enc.c:178-187).  Returns bytes written. */
int gm_encode_frame(gm_encoder *e, const uint8_t *luma, const uint8_t *chroma, uint8_t *out, int out_cap);
void gm_close(gm_encoder *e);

/* Intermediates of the most recent frame (for kernel-level parity tests). */
int gm_coded_width(const gm_encoder *e);
int gm_coded_height(const gm_encoder *e);
const gm_mb *gm_mbs(const gm_encoder *e);
const uint8_t *gm_recon(const gm_encoder *e, int plane);       /* after deblocking */
const uint8_t *gm_recon_unfiltered(const gm_encoder *e, int plane);
const uint8_t *gm_source(const gm_encoder *e, int plane);      /* ingested (padded, planar) */
int gm_last_frame_type(const gm_encoder *e);                   /* 1 = I, 0 = P */
/* Position of the next frame inside its GOP (cedar.c:118 frame_p_count; 0 = the next frame is an IDR picture).  For
 * callers that own the GOP counter themselves: oracle/refsim's model of the video engine is told the picture type per
 * frame by the reference driver's PARA0 write (cedar.c:1160-1163). */
void gm_set_frame_p_count(gm_encoder *e, int frame_p_count);
double gm_last_sse_y(const gm_encoder *e);

/* Header writer on its own (for byte-identity tests against Appendix A vectors). */
int gm_write_sps(const gm_config *cfg, uint8_t *out, int cap);
int gm_write_pps(const gm_config *cfg, uint8_t *out, int cap);
/* Writes start code + NAL header + slice header bits; *nbits = header bits after NAL byte. */
int gm_slice_header_bits(int frame_i, int frame_p_count, int cabac, uint32_t *bits, int *nbits);
/* The same with first_mb_in_slice != 0 (slice_rows extension); up to 64 bits. */
int gm_slice_header_bits64(int frame_i, int frame_p_count, int cabac, int first_mb, uint64_t *bits, int *nbits);

/* The CABAC arithmetic coder on its own (for kernel-level tests of the product's coder): one slice's RBSP from the
 * bins of the product's format (ctxIdx 0..459 in bits 0..9, 1 << 10 bypass, 1 << 11 terminate, value in bit 15; the
 * last bin and only it is terminate(1)) coded in the initial states of (frame_i, qp) after hdr_nbits header bits.
 * Returns the RBSP bytes written to out, -EINVAL for a malformed bin array, -ENOMEM when cap is too small.  Optional:
 * pre[i] = the state (pStateIdx << 1 | valMPS) regular bin i was coded in; stats[0] = the longest run of outstanding
 * bits, stats[1] = the bit that ended it (1 = a carry), stats[2] = slice data bits through the rbsp stop bit. */
int gm_cabac_code_bins(const uint16_t *bins, int n, int frame_i, int qp, uint64_t hdr_bits, int hdr_nbits, uint8_t *out,
                       int cap, uint8_t *pre, int *stats);

/* Deterministic synthetic moving-pattern clip (integer only, stateless per pixel). */
void gm_synth_frame(int width, int height, int format, int t, uint8_t *luma, uint8_t *chroma);

#ifdef __cplusplus
}
#endif
#endif
