/*
 * cedar_b200 -- C ABI of the B200-native drop-in for libv/cedarx_h264_encoder's encode path.
 *
 * The reference's userspace talks to the Allwinner Cedar VE through two ioctls and three mmaps
 * (/root/reference/kernel/cedar_ioctl.h:7-46, userspace/h264enc.c:47-117,178-198).  This header
 * is what a maintainer binds instead; every entry point cites the interface it replaces.
 * Plain C: pointers and sizes only.  All buffers are owned by the library (as the kernel owns
 * the DMA buffers in the reference); the caller never frees them.
 *
 * There is NO CPU fallback: every encode call runs hand-written sm_100a CUDA kernels and fails
 * with a negative errno if no CUDA device is usable.
 */
#ifndef CEDAR_B200_H
#define CEDAR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CEDAR_B200_FORMAT_NV12 0 /* CEDAR_IOCTL_CONFIG_FORMAT_NV12, cedar_ioctl.h:15 */
#define CEDAR_B200_FORMAT_NV16 1 /* CEDAR_IOCTL_CONFIG_FORMAT_NV16, cedar_ioctl.h:16 */
#define CEDAR_B200_ENTROPY_CAVLC 0 /* CEDAR_IOCTL_ENTROPY_CODING_CAVLC, cedar_ioctl.h:30 */
#define CEDAR_B200_ENTROPY_CABAC 1 /* CEDAR_IOCTL_ENTROPY_CODING_CABAC, cedar_ioctl.h:31 */

/*
 * Replaces the input half of struct cedar_ioctl_config (cedar_ioctl.h:12-32): same field names,
 * same meaning, same validation (kernel/cedar.c:744-789).  Fields after entropy_coding_mode are
 * extensions; zero means "reference behaviour / default".
 */
struct cedar_b200_config {
    int src_width;
    int src_height;
    int src_format;
    int dst_width;
    int dst_height;
    int profile;
    int level;
    int qp;
    int keyframe_interval;
    int thumbnail;           /* accepted and reported back as 0: the ISP thumbnail scaler is out of scope */
    int thumbnail_downscale;
    int entropy_coding_mode;
    /* extensions */
    int me_range;            /* integer-pel full-search radius, 1..64; 0 = 16 */
    int relax_gop;           /* non-zero: accept keyframe_interval >= 32 (cedar.c:784-789 rejects it) */
    int device;              /* CUDA device ordinal */
    int gops_in_flight;      /* clip mode: closed GOPs encoded concurrently on this GPU; 0 = auto */
    int max_clip_frames;     /* clip mode: capacity of the clip buffers in frames; 0 = clip mode off */
    int slice_rows;          /* macroblock rows per slice; 0 = one slice per picture as the reference writes it
                              * (first_mb_in_slice always 0, cedar.c:992-993).  N > 0: every N rows start a new slice
                              * NAL, coded by its own (parallel) entropy coder at some cost in bits. */
    int sps_crop;            /* non-zero: signal src_width x src_height with frame cropping in the SPS (1920x1080 instead
                              * of the coded 1920x1088).  The reference never does: cedar.c:756-761 makes :924-931 dead. */
    int auto_level;          /* non-zero: level_idc = lowest level whose MaxFS fits the picture (4K: 5.1) instead of the
                              * configured `level`, which the reference writes unchecked (cedar.c:900). */
    int repeat_headers;      /* non-zero: SPS + PPS in front of every IDR picture, so that every closed GOP (e.g. one
                              * GPU's share of a GOP-parallel encode) decodes on its own; the reference writes them
                              * once, before the first frame (cedar.c:1058-1061). */
    int intra4x4;            /* non-zero: I frames may use Intra4x4 macroblocks (nine prediction modes per 4x4 block)
                              * where their SAD-based cost beats the best Intra16x16 mode. */
    int p_intra;             /* non-zero: macroblocks of P frames are coded as Intra16x16 where that beats the motion
                              * search (scene changes, uncovered content). */
    int queue_gops;          /* non-zero: QUEUED mode of the per-frame call (SURVEY 8b).  encode_frame() keeps the
                              * reference's call pattern -- fill the input buffers, call, write `ret` bytes
                              * (userspace/h264enc.c:181-198) -- but the frames are encoded GOP-parallel in batches of
                              * queue_gops closed GOPs: the call returns 0 while the first two batches fill, afterwards
                              * the bytes of frame t - 2 * queue_gops * keyframe_interval, and cedar_b200_flush() drains
                              * the rest, one frame per call.  The concatenated output is byte-identical to the
                              * synchronous mode. */
};

/*
 * Replaces the output half of struct cedar_ioctl_config (cedar_ioctl.h:34-45) and the three
 * mmap() calls of userspace/h264enc.c:76-106: host pointers (pinned memory) instead of DMA
 * addresses.  The caller fills input_luma / input_chroma before every encode_frame call and
 * reads `ret` bytes from bytestream after it (userspace/h264enc.c:181-197).
 */
struct cedar_b200_io {
    void *input_luma;
    int input_luma_size;   /* src_width * src_height rounded up to 4096 (cedar.c:610-615) */
    void *input_chroma;
    int input_chroma_size; /* NV12: w*h/2, NV16: w*h, rounded up to 4096 (cedar.c:621-624) */
    void *bytestream;
    int bytestream_size;   /* worst-case frame; the reference's fixed 1 MiB (cedar.c:663) is too small for 4K */
};

/* One handle = one stream of work on one GPU (the reference: one opener of /dev/cedar_dev, kernel/cedar.c:457-474).
 * A handle is not thread-safe, but different handles share nothing and every call selects its handle's device, so
 * handles may be driven from different host threads -- two or three per GPU keep the GPU full (INTEGRATION.md 4). */
typedef struct cedar_b200_handle cedar_b200_handle;

/* open("/dev/cedar_dev") + ioctl(CEDAR_IOCTL_CONFIG) + 3x mmap (userspace/h264enc.c:149,68,76-106;
 * kernel/cedar.c:457-474,732-866).  Returns 0 or -EINVAL / -ENOMEM / -ENODEV. */
int cedar_b200_open(const struct cedar_b200_config *cfg, struct cedar_b200_io *io, cedar_b200_handle **h);

/* ioctl(CEDAR_IOCTL_ENCODE) (kernel/cedar.c:1032-1209): synchronous; encodes the frame currently in
 * io->input_luma / io->input_chroma; returns the number of bytes now valid at io->bytestream
 * (SPS+PPS precede the first frame only, cedar.c:1058-1061) or a negative errno. */
int cedar_b200_encode_frame(cedar_b200_handle *h);

/* Queued mode only (cfg.queue_gops != 0): after the last encode_frame() call, every call returns the bytes of the next
 * outstanding frame in io->bytestream (display order), 0 when the stream is drained, or a negative errno.  In the
 * synchronous mode it returns 0: nothing is ever outstanding. */
int cedar_b200_flush(cedar_b200_handle *h);

/* close(fd) -> cedar_slashdev_release (kernel/cedar.c:706-730): frees everything and prints the
 * busy/total time line the reference prints. */
void cedar_b200_close(cedar_b200_handle *h);

/* ---------------------------------------------------------------------------------------------
 * Clip mode (the queued / GOP-parallel path of SURVEY 8b): a whole clip is encoded with several
 * closed GOPs in flight.  Output is byte-identical to calling encode_frame once per frame.
 * ------------------------------------------------------------------------------------------- */

/* Pinned host staging for `max_clip_frames` packed input frames (luma then chroma, back to back,
 * exactly the bytes the reference's read loop consumes per frame, userspace/h264enc.c:181-187). */
void *cedar_b200_clip_input(cedar_b200_handle *h, size_t *frame_bytes);

/* Host -> device copy of the first nframes of the staging area.  Asynchronous, and paced by the encode that follows:
 * the copies of a pass are issued by cedar_b200_clip_encode, one pass ahead of the pass that consumes them, so that
 * several handles share the copy engine frame by frame, not clip by clip.  The staging area must not be written again
 * before the cedar_b200_clip_download (or cedar_b200_stats) of that encode has returned. */
int cedar_b200_clip_upload(cedar_b200_handle *h, int nframes);

/* Encode nframes already resident in device memory; frame `first_frame_index + i` of the stream
 * (this decides which frames are IDR and whether SPS/PPS are emitted: only before stream frame 0).
 * Leaves the packed Annex-B stream in device memory.  Returns 0 or a negative errno. */
int cedar_b200_clip_encode(cedar_b200_handle *h, int nframes, int first_frame_index);

/* Device -> host copy of the packed stream.  *out receives a pointer to pinned host memory valid
 * until the next clip call; frame_bytes (may be NULL) receives nframes per-frame byte counts.
 * Returns total bytes or a negative errno.  The entropy buffers of clip mode are sized by a heuristic bound
 * per macroblock; if the coded clip exceeds it, this call enlarges them and encodes the (still resident)
 * clip again before it returns -- the caller sees the bytes, and a note on stderr. */
long long cedar_b200_clip_download(cedar_b200_handle *h, const uint8_t **out, int *frame_bytes);

/* Statistics of the last encode_frame / clip_encode: sum of squared luma error per frame
 * (for Y-PSNR) -- sse_y must hold nframes doubles. */
int cedar_b200_stats(cedar_b200_handle *h, double *sse_y, int nframes);

/* Per-kernel device timing of the work issued since the last call with reset != 0.
 * enable = 1: every launch is bracketed by CUDA events on the stream it is launched on (live, overlapped);
 * enable = 2: additionally all work is issued on one stream, so the event times are standalone kernel times;
 * enable = 3: as 2, with the measurement builds of the kernels: work counters (debug_read 8) and, if CEDAR_B200_NO_PRUNE was
 *             set at open(), a motion search without pruning.  Same bytes, slower kernels: never time the product this way.
 * names/ms/launches hold up to `cap` entries; returns the number of kernel classes. */
int cedar_b200_profile_enable(cedar_b200_handle *h, int enable);
int cedar_b200_profile_read(cedar_b200_handle *h, const char **names, float *ms, int *launches, int cap, int reset);

/* The CUDA stream (cudaStream_t) every kernel and copy of this handle is issued on, so a caller can
 * bracket calls with its own CUDA events. */
void *cedar_b200_stream(cedar_b200_handle *h);

/* Total kernels launched by this handle so far (bench.py's gpu_launches). */
long long cedar_b200_launch_count(cedar_b200_handle *h);

/* Debug / parity-test access to intermediates of the last encode_frame call (lane 0):
 * what = 0 source planes, 1 unfiltered recon, 2 deblocked recon (Y then U then V, coded size),
 *        3 macroblock info records, 4 nnz records, 5 coefficient levels,
 *        6 CABAC bins per slice NAL of the last call (uint32 each), 7 Intra4x4 prediction modes (16 bytes per
 *        macroblock), 8 measurement counters of the work issued while profiling was on (520 uint64: [0] executed
 *        VABSDIFF4 lane-instructions of the motion search, [8 + c] CABAC bins of context c).  Returns bytes copied. */
long long cedar_b200_debug_read(cedar_b200_handle *h, int what, void *dst, size_t cap);

/* Header writer on its own (host C; restates kernel/cedar.c:868-1030) for byte-identity tests. */
int cedar_b200_write_sps(const struct cedar_b200_config *cfg, uint8_t *out, int cap);
int cedar_b200_write_pps(const struct cedar_b200_config *cfg, uint8_t *out, int cap);
int cedar_b200_slice_header(int frame_i, int frame_p_count, int cabac, uint32_t *bits, int *nbits);
/* Slice header of a slice that starts at macroblock first_mb (slice_rows extension); up to 64 bits. */
int cedar_b200_slice_header_mb(int frame_i, int frame_p_count, int cabac, int first_mb, uint64_t *bits, int *nbits);

/* ---------------------------------------------------------------------------------------------
 * Ordered pipeline over several handles and GPUs (csrc/pipeline.cpp): the north star's "GOP-parallel across the GPUs of
 * one box, per-GPU bytestreams concatenated on the host".  Batches of gops_per_batch closed GOPs; batch b is encoded by
 * worker b % W, W = ndevices * handles_per_device, every worker being one handle on one device with its own host
 * thread.  The batches come back in submission order and concatenate to exactly the stream one handle -- or the
 * frame-at-a-time call -- produces: SPS + PPS only in front of stream frame 0 (kernel/cedar.c:1058-1061), an IDR
 * picture at every multiple of keyframe_interval (:1047-1050, :1193-1196).
 * One producer thread (acquire, fill, submit, ..., finish) and one consumer thread (next, ...), which may be the same
 * thread as long as it does not acquire more than W batches ahead of what it has consumed.
 * ------------------------------------------------------------------------------------------- */
typedef struct cedar_b200_pipe cedar_b200_pipe;

/* devices == NULL or ndevices == 0: cfg->device only.  handles_per_device == 0: 2.  gops_per_batch == 0: 4.
 * cfg->max_clip_frames and cfg->device are overridden per worker.  Returns 0 or a negative errno. */
int cedar_b200_pipe_open(const struct cedar_b200_config *cfg, const int *devices, int ndevices, int handles_per_device,
                         int gops_per_batch, cedar_b200_pipe **p);
int cedar_b200_pipe_workers(cedar_b200_pipe *p);
/* Pinned host staging of the next batch: capacity_frames packed frames of frame_bytes each (luma then chroma, as the
 * reference's read loop consumes them, userspace/h264enc.c:181-187).  Blocks until the worker that will encode the
 * batch is free (its previous batch consumed).  NULL when a batch is already being filled, after a short batch (it ends
 * the stream) or after finish. */
void *cedar_b200_pipe_acquire(cedar_b200_pipe *p, size_t *frame_bytes, int *capacity_frames);
/* Hands the acquired batch, holding nframes frames, to its worker (asynchronous).  Only the last batch of a stream may
 * hold fewer than capacity_frames; nframes == 0 gives the buffer back and ends the stream. */
int cedar_b200_pipe_submit(cedar_b200_pipe *p, int nframes);
/* No more batches will be submitted: pipe_next returns 0 once everything submitted has been consumed. */
int cedar_b200_pipe_finish(cedar_b200_pipe *p);
/* The next batch in submission order: total bytes (> 0), the packed stream in *out, per-frame byte counts, frame count
 * and per-frame luma SSE (pointers valid until the next pipe_next / pipe_release call).  wait != 0 blocks until that
 * batch is encoded; otherwise -EAGAIN.  0: nothing outstanding.  Negative errno: that batch failed. */
long long cedar_b200_pipe_next(cedar_b200_pipe *p, const uint8_t **out, const int **frame_sizes, int *nframes,
                               const double **sse_y, int wait);
/* The consumer is done with the batch the last pipe_next returned (implied by the next pipe_next call). */
int cedar_b200_pipe_release(cedar_b200_pipe *p);
void cedar_b200_pipe_close(cedar_b200_pipe *p);

const char *cedar_b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* CEDAR_B200_H */
