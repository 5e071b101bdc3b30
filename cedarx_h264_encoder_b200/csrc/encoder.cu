// Host layer of the B200 H.264 encoder: the C ABI of include/cedar_b200.h.
//
// Mirrors the reference's driver control flow with kernel launches in place of register writes:
//   cedar_slashdev_ioctl_config  (kernel/cedar.c:732-866)  -> cedar_b200_open
//   cedar_buffers_init           (kernel/cedar.c:605-704)  -> alloc_buffers (cudaMalloc / pinned host)
//   cedar_slashdev_ioctl_encode  (kernel/cedar.c:1032-1209) -> cedar_b200_encode_frame / clip_encode
//   cedar_slashdev_release       (kernel/cedar.c:706-730)  -> cedar_b200_close
// There is no CPU fallback: without a CUDA device open() fails with -ENODEV.
#include "../../include/cedar_b200.h"
#include "cedar_headers.h"
#include "kernels.cuh"

#include <cuda_runtime.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <errno.h>
#include <vector>

using namespace cedar;

#define ALIGN_UP(x, a) (((x) + ((a)-1)) & ~((size_t)(a)-1))

namespace {

enum KernelId {
    K_INGEST, K_ME, K_INTER, K_PINTRA, K_INTRA, K_BS, K_DEBLOCK, K_SSE, K_ESIZE, K_ESCAN, K_EZERO, K_EWRITE,
    K_CRESOLVE, K_CCODE, K_EPBCOUNT, K_EPBSCAN, K_PACKSCAN, K_EPBWRITE, K_COUNT
};
const char *kKernelNames[K_COUNT] = {
    "ingest_kernel", "me_kernel", "inter_kernel", "pintra_decide_kernel", "intra_kernel", "bs_kernel", "deblock_kernel",
    "sse_kernel", "entropy_size_kernel", "entropy_scan_kernel", "rbsp_zero_kernel", "entropy_write_kernel",
    "cabac_resolve_kernel", "cabac_code_kernel", "epb_count_kernel", "epb_scan_kernel", "pack_scan_kernel", "epb_write_kernel"};

const uint8_t kChromaQp[52] = {0,  1,  2,  3,  4,  5,  6,  7,  8,  9,  10, 11, 12, 13, 14, 15, 16, 17,
                               18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 29, 30, 31, 32, 32, 33,
                               34, 34, 35, 35, 36, 36, 37, 37, 37, 38, 38, 38, 39, 39, 39, 39};

struct ProfEntry {
    int id;
    cudaEvent_t a, b;
};

} // namespace

__global__ void rbsp_zero_kernel(Step s, uint8_t *rbsp, unsigned rbsp_cap, const uint32_t *rbsp_len)
{
    int f = lane_frame(s, blockIdx.y);
    if (f < 0)
        return;
    const size_t u = (size_t)f * gridDim.z + blockIdx.z; // blockIdx.z = slice
    size_t words = ((size_t)rbsp_len[u] + 8 + 3) / 4;
    uint32_t *p = (uint32_t *)(rbsp + u * rbsp_cap);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < words; i += (size_t)gridDim.x * blockDim.x)
        p[i] = 0;
}

struct cedar_b200_handle {
    cedar_b200_config cfg;
    Geom g;
    int K;                 // keyframe_interval
    int F;                 // clip capacity in frames (>= 1)
    bool clip_mode;        // max_clip_frames > 0: the clip calls are usable and the buffers are sized for whole clips
    int L;                 // lanes (GOPs in flight)
    int S;                 // slices per picture (1 = the reference's layout)
    size_t raw_frame_bytes;
    cudaStream_t stream;      // recon + parallel entropy stages
    // serial CABAC stages run on a pool of side streams so that the coders of successive steps overlap
    // each other and the following frames' reconstruction
    enum { NSIDE = 32 };
    cudaStream_t stream_cabac[NSIDE];
    // Per step only ME -> residual -> deblock stay on the main stream.  Ingest runs one step ahead on
    // stream_pre, SSE and the parallel entropy passes one step behind on stream_post; source planes and
    // syntax records are double buffered (index = step parity) so the three can overlap.
    cudaStream_t stream_pre, stream_post;
    cudaEvent_t ev_ingest[2], ev_main[2], ev_post[2], ev_begin, ev_post_done;
    cudaEvent_t ev_syn[2], ev_ent[2]; // syntax records of step parity p final (after bs_kernel) / its entropy passes done
    bool post_valid[2]; // ev_post[p] has been recorded in this stream of work
    // clip upload: host->device copies run on their own stream in step order; step t waits for ev_upload[t] only
    cudaStream_t stream_copy;
    std::vector<cudaEvent_t> ev_upload;
    cudaEvent_t ev_encode_done;
    bool upload_pending;
    // Paced upload (D = CEDAR_B200_UPLOAD_AHEAD, default 1): clip_upload only notes the request; clip_encode issues the
    // copies of pass j + D behind the ingest of pass j, so that at most D passes of this handle are queued on the copy
    // engine and the first frames of another handle's next clip are not stuck behind a whole clip of copies (the copy
    // engine serves copies in issue order).  Measured, three handles, 1080p end to end: D = 0 (all copies at once)
    // 12 050-12 600 frames/s, D = 1 13 000-13 700, D = 2 12 660-12 770, D = 8 12 720; device resident 14 000.
    int upload_ahead, upload_deferred_n;
    cudaEvent_t ev_cabac[NSIDE];
    unsigned side_used; // bit i: side stream i has work the main stream has not joined yet
    int side_next;
    int grow;             // multiplier on the heuristic entropy-buffer bounds; clip mode raises it and re-encodes on overflow
    int last_first_frame; // of the last clip_encode
    int device; // every entry point selects it: the current device is per host thread, and handles are driven from threads

    // cedar.c:118-119 counters and the ping-pong reference (frame mode, lane 0)
    int frame_p_count, frame_count;

    // pinned host
    uint8_t *h_in_luma, *h_in_chroma, *h_bytestream;
    int in_luma_size, in_chroma_size, bytestream_size;
    uint8_t *h_clip_in, *h_clip_out;
    size_t out_cap;
    int *h_frame_bytes;
    unsigned long long *h_total;
    unsigned long long *h_sse;
    int *h_error;

    // device
    uint8_t *d_raw, *d_src[2], *d_unf, *d_rec[2];
    MbInfo *d_mbi[2];
    uint8_t *d_nnz[2];
    uint8_t *d_i4[2]; // Intra4x4 prediction modes, [L][nmb][16]
    uint8_t *d_pwant; // p_intra: macroblocks of the current P step to re-code as intra, [L][nmb]
    int *d_pcount;    // p_intra: how many per lane
    int16_t *d_coef[2];
    int *d_flags; // [3][L][mbh]
    uint32_t *d_me_tabs; // me_kernel's cost / task tables (me_build_tables)
    unsigned long long *d_counters; // measurement (profiling on): [0, 5) me_kernel (MeShape::exec_count), [8 + c] bins of context c
    bool no_prune;                  // measurement (CEDAR_B200_NO_PRUNE at open): the search accumulates every candidate to the end
    uint8_t *d_bs; // [L][nmb][32] boundary strengths
    unsigned long long *d_sse;
    EntropyBufs eb;
    unsigned long long *d_hdr_bits;
    int *d_hdr_nbits;
    uint32_t *d_chunk_cnt, *d_nal_bytes;
    unsigned chunks_per_frame; // per slice NAL
    unsigned long long *d_nal_off, *d_total;
    int *d_frame_bytes;
    uint8_t *d_out;
    uint8_t prefix[64];
    int prefix_len;

    int last_nframes, last_cur, last_par;
    bool sse_valid; // h_sse holds the statistics of the last encode
    // Queued mode of the per-frame call (cfg.queue_gops): this handle is only a front -- io buffers and counters -- over a
    // pipeline of worker handles (pipeline.cpp); none of the device members above exist.
    cedar_b200_pipe *pipe;
    uint8_t *q_staging;        // batch being filled (pipe_acquire)
    size_t q_frame_bytes;
    int q_cap, q_fill;         // frames per batch, frames in the batch being filled
    long long q_in, q_out;     // frames accepted / returned so far
    std::vector<uint8_t> q_bytes; // coded bytes of the batch being handed out, one frame per call
    std::vector<int> q_sizes;
    std::vector<double> q_sse;
    size_t q_pos, q_off;
    long long launches;
    bool prof;
    bool serialize; // profile mode 2: no stream overlap, so that per-kernel event times are standalone times
    bool count;     // profile mode 3: mode 2 with the measurement builds of the kernels (work counters, CEDAR_B200_NO_PRUNE)
    std::vector<ProfEntry> prof_pending;
    std::vector<cudaEvent_t> ev_pool;
    float prof_ms[K_COUNT];
    int prof_n[K_COUNT];
    std::chrono::steady_clock::time_point t_open;
    double busy_ns;
};

namespace {

#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) {                                                                       \
            fprintf(stderr, "cedar_b200: %s failed: %s (%s:%d)\n", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return -EIO;                                                                               \
        }                                                                                              \
    } while (0)

cudaEvent_t get_event(cedar_b200_handle *h)
{
    if (!h->ev_pool.empty()) {
        cudaEvent_t e = h->ev_pool.back();
        h->ev_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

struct LaunchScope {
    cedar_b200_handle *h;
    cudaStream_t st;
    ProfEntry pe;
    LaunchScope(cedar_b200_handle *hh, int id, cudaStream_t s) : h(hh), st(s)
    {
        pe.id = id;
        h->launches++;
        if (h->prof) {
            pe.a = get_event(h);
            pe.b = get_event(h);
            cudaEventRecord(pe.a, st);
        }
    }
    ~LaunchScope()
    {
        if (h->prof) {
            cudaEventRecord(pe.b, st);
            h->prof_pending.push_back(pe);
        }
    }
};

#define LAUNCH_ON(st, id, kern, grid, block, smem, ...)                                                      \
    do {                                                                                                     \
        {                                                                                                    \
            LaunchScope ls_(h, id, st);                                                                      \
            kern<<<grid, block, smem, st>>>(__VA_ARGS__);                                                    \
        }                                                                                                    \
        cudaError_t le_ = cudaGetLastError();                                                                \
        if (le_ != cudaSuccess) {                                                                            \
            fprintf(stderr, "cedar_b200: launch of %s failed: %s\n", kKernelNames[id], cudaGetErrorString(le_)); \
            return -EIO;                                                                                     \
        }                                                                                                    \
    } while (0)
#define LAUNCH(id, kern, grid, block, smem, ...) LAUNCH_ON(h->stream, id, kern, grid, block, smem, __VA_ARGS__)

void prof_collect(cedar_b200_handle *h)
{
    cudaStreamSynchronize(h->stream);
    for (int i = 0; i < cedar_b200_handle::NSIDE; i++)
        cudaStreamSynchronize(h->stream_cabac[i]);
    // CEDAR_B200_TIMELINE=<file> (diagnosis): start/end of every launch relative to the first one
    FILE *tl = nullptr;
    if (const char *path = getenv("CEDAR_B200_TIMELINE"))
        if (!h->prof_pending.empty())
            tl = fopen(path, "a");
    for (auto &pe : h->prof_pending) {
        float ms = 0;
        cudaEventElapsedTime(&ms, pe.a, pe.b);
        if (tl) {
            float t0 = 0;
            cudaEventElapsedTime(&t0, h->prof_pending.front().a, pe.a);
            fprintf(tl, "%s,%.4f,%.4f\n", kKernelNames[pe.id], t0, t0 + ms);
        }
        h->prof_ms[pe.id] += ms;
        h->prof_n[pe.id]++;
        h->ev_pool.push_back(pe.a);
        h->ev_pool.push_back(pe.b);
    }
    if (tl)
        fclose(tl);
    h->prof_pending.clear();
}

int validate(const cedar_b200_config *c) // kernel/cedar.c:744-789, same order, same -EINVAL
{
    if ((c->src_width & 0x01) || (c->src_height & 0x01)) {
        fprintf(stderr, "cedar_b200: src width %d, height %d not aligned.\n", c->src_width, c->src_height);
        return -EINVAL;
    }
    if ((c->dst_width & 0x0F) || (c->dst_height & 0x0F)) {
        fprintf(stderr, "cedar_b200: dst width %d, height %d not aligned.\n", c->dst_width, c->dst_height);
        return -EINVAL;
    }
    if ((c->src_width > c->dst_width) || (c->src_height > c->dst_height)) {
        fprintf(stderr, "cedar_b200: src (%d,%d) > dst (%d, %d)\n", c->src_width, c->src_height, c->dst_width,
                c->dst_height);
        return -EINVAL;
    }
    if ((c->qp <= 0) || (c->qp > 47)) {
        fprintf(stderr, "cedar_b200: invalid QP %d\n", c->qp);
        return -EINVAL;
    }
    if ((c->src_format != CEDAR_B200_FORMAT_NV12) && (c->src_format != CEDAR_B200_FORMAT_NV16)) {
        fprintf(stderr, "cedar_b200: invalid color format.\n");
        return -EINVAL;
    }
    if ((c->keyframe_interval <= 0) || (c->keyframe_interval >= 32 && !c->relax_gop)) {
        fprintf(stderr, "cedar_b200: invalid keyframe interval %d\n", c->keyframe_interval);
        return -EINVAL;
    }
    if (c->src_width <= 0 || c->src_height <= 0 || c->me_range < 0 || c->me_range > 64 || c->max_clip_frames < 0 ||
        c->gops_in_flight < 0 || c->slice_rows < 0) {
        fprintf(stderr, "cedar_b200: invalid extension field.\n");
        return -EINVAL;
    }
    return 0;
}

template <class T> int dmalloc(T **p, size_t n)
{
    cudaError_t e = cudaMalloc((void **)p, n * sizeof(T));
    if (e != cudaSuccess) {
        cudaGetLastError(); // not sticky, but it would surface at the next launch check of any handle
        fprintf(stderr, "cedar_b200: cudaMalloc(%zu) failed: %s\n", n * sizeof(T), cudaGetErrorString(e));
        return -ENOMEM;
    }
    return 0;
}
template <class T> int hmalloc(T **p, size_t n)
{
    cudaError_t e = cudaHostAlloc((void **)p, n * sizeof(T), cudaHostAllocDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        fprintf(stderr, "cedar_b200: cudaHostAlloc(%zu) failed: %s\n", n * sizeof(T), cudaGetErrorString(e));
        return -ENOMEM;
    }
    return 0;
}

// The buffers whose size is a heuristic bound on the coded size (RBSP per slice NAL, CABAC bin pool, limb scratch,
// emulation-prevention chunk counters, packed output on device and host).  h->grow scales the bounds: clip mode raises
// it and encodes again when a clip overflows them (clip_download), frame mode reports the overflow.
void free_entropy_buffers(cedar_b200_handle *h)
{
    void *dev[] = {h->eb.rbsp, h->eb.bins, h->eb.limbs, h->d_chunk_cnt, h->d_out};
    for (void *p : dev)
        if (p)
            cudaFree(p);
    if (h->h_clip_out)
        cudaFreeHost(h->h_clip_out);
    h->eb.rbsp = nullptr, h->eb.bins = nullptr, h->eb.limbs = nullptr, h->d_chunk_cnt = nullptr, h->d_out = nullptr;
    h->h_clip_out = nullptr;
}

int alloc_entropy_buffers(cedar_b200_handle *h)
{
    const Geom &g = h->g;
    const int F = h->F, L = h->L, S = h->S;
    const size_t U = (size_t)F * S, grow = (size_t)h->grow; // U slice NALs
    const size_t slice_mbs = (size_t)g.srows * g.mbw;
    int r = 0;
    const bool clip = h->clip_mode;
    // all bounds in 64 bits: the x4 regrow of clip mode reaches 8 GB per slice at 4K before anything else gives up
    const size_t rbsp_cap = ALIGN_UP(slice_mbs * (clip ? (g.qp < 20 ? 1024 : 400) : 1024) * grow + 4096, 256);
    size_t per_frame_out =
        (clip ? (size_t)g.nmb * (g.qp < 20 ? 512 : 96) * grow + 4096 : (size_t)h->bytestream_size) + 8 * S + 64;
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    if (rbsp_cap > 0xFFFFFF00ull || rbsp_cap * U > total_b || per_frame_out * F > total_b) {
        fprintf(stderr, "cedar_b200: entropy buffers of %zu bytes per slice x %zu slices do not fit the device\n", rbsp_cap, U);
        return -ENOMEM;
    }
    h->eb.rbsp_cap = (unsigned)rbsp_cap;
    h->out_cap = per_frame_out * F;
    size_t bins_per_mb = clip ? (g.qp < 12 ? 8192 : (g.qp < 20 ? 2048 : 640)) : 16384;
    // the pool is shared by all frames of a clip (bump allocation), so for long clips the per-macroblock allowance can
    // shrink: at most 24 GB, at least 160 bins per macroblock (the 1080p benchmark clip averages 38, its I frames 145)
    if (clip && bins_per_mb * g.nmb * F * sizeof(uint16_t) > (24ull << 30)) {
        bins_per_mb = (24ull << 30) / ((size_t)g.nmb * F * sizeof(uint16_t));
        if (bins_per_mb < 160)
            bins_per_mb = 160;
    }
    if (const char *e = getenv("CEDAR_B200_BINS_PER_MB"))
        bins_per_mb = (size_t)atoll(e);
    bins_per_mb *= grow;
    h->eb.bins_cap = g.cabac ? (unsigned long long)(bins_per_mb * g.nmb + 8) * F + 64 : 0;
    h->eb.limb_cap = h->eb.rbsp_cap / 2 + 8;
    h->chunks_per_frame = (h->eb.rbsp_cap + EPB_CHUNK - 1) / EPB_CHUNK;
    if (clip)
        r |= hmalloc(&h->h_clip_out, h->out_cap);
    r |= dmalloc(&h->eb.rbsp, (size_t)h->eb.rbsp_cap * U);
    if (g.cabac) {
        r |= dmalloc(&h->eb.bins, (size_t)h->eb.bins_cap + 64); // + slack: 16-byte vector loads round outwards
        // one region per side stream; frame mode finishes every frame before the next one starts: one region
        r |= dmalloc(&h->eb.limbs, (size_t)h->eb.limb_cap * L * S * (clip ? cedar_b200_handle::NSIDE : 1));
    }
    r |= dmalloc(&h->d_chunk_cnt, (size_t)h->chunks_per_frame * U);
    r |= dmalloc(&h->d_out, h->out_cap + 64);
    return r;
}

int alloc_buffers(cedar_b200_handle *h)
{
    const Geom &g = h->g;
    const int F = h->F, L = h->L;
    int r = 0;
    // frame-mode I/O, sized like cedar_buffers_init (cedar.c:610-624) but in pinned host memory
    h->in_luma_size = (int)ALIGN_UP((size_t)g.src_w * g.src_h, 4096);
    size_t chroma_bytes = (size_t)g.src_w * g.src_h / (g.src_format == CEDAR_B200_FORMAT_NV16 ? 1 : 2);
    h->in_chroma_size = (int)ALIGN_UP(chroma_bytes, 4096);
    h->bytestream_size = (int)ALIGN_UP((size_t)g.nmb * 1536 + 4096, 4096);
    r |= hmalloc(&h->h_in_luma, h->in_luma_size);
    r |= hmalloc(&h->h_in_chroma, h->in_chroma_size);
    r |= hmalloc(&h->h_bytestream, h->bytestream_size);
    r |= hmalloc(&h->h_frame_bytes, F);
    r |= hmalloc(&h->h_total, 1);
    r |= hmalloc(&h->h_sse, F);
    r |= hmalloc(&h->h_error, 1);
    if (r)
        return r;

    const int S = h->S;
    const size_t U = (size_t)F * S; // slice NALs
    if (h->clip_mode)
        r |= hmalloc(&h->h_clip_in, h->raw_frame_bytes * F);
    r |= dmalloc(&h->d_raw, h->raw_frame_bytes * F + 64);
    r |= dmalloc(&h->d_src[0], g.frame_bytes * L);
    r |= dmalloc(&h->d_src[1], g.frame_bytes * L);
    r |= dmalloc(&h->d_unf, g.frame_bytes * L);
    r |= dmalloc(&h->d_rec[0], g.frame_bytes * L);
    r |= dmalloc(&h->d_rec[1], g.frame_bytes * L);
    for (int p = 0; p < 2; p++) {
        r |= dmalloc(&h->d_mbi[p], (size_t)g.nmb * L);
        r |= dmalloc(&h->d_nnz[p], (size_t)g.nmb * L * NNZ_STRIDE);
        r |= dmalloc(&h->d_i4[p], (size_t)g.nmb * L * 16);
        r |= dmalloc(&h->d_coef[p], (size_t)g.nmb * L * COEF_STRIDE);
    }
    r |= dmalloc(&h->d_flags, (size_t)3 * L * g.mbh);
    r |= dmalloc(&h->d_me_tabs, me_table_words(g.R, me_strip(g.R)));
    r |= dmalloc(&h->d_counters, 8 + 512);
    r |= dmalloc(&h->d_pwant, (size_t)g.nmb * L);
    r |= dmalloc(&h->d_pcount, (size_t)L);
    r |= dmalloc(&h->d_bs, (size_t)g.nmb * L * 32);
    r |= dmalloc(&h->d_sse, F);
    r |= dmalloc(&h->eb.mb_size, (size_t)L * (g.nmb + S + 1));
    r |= dmalloc(&h->eb.mb_off, (size_t)L * (g.nmb + S + 1));
    r |= dmalloc(&h->d_hdr_bits, (size_t)(F > h->K ? F : h->K) * S);
    r |= dmalloc(&h->d_hdr_nbits, (size_t)(F > h->K ? F : h->K) * S);
    r |= dmalloc(&h->eb.rbsp_len, U);
    r |= dmalloc(&h->eb.bins_cursor, 1);
    r |= dmalloc(&h->eb.bins_off, U);
    r |= dmalloc(&h->eb.bins_len, U);
    r |= dmalloc(&h->eb.error, 1);
    r |= dmalloc(&h->d_nal_bytes, U);
    r |= dmalloc(&h->d_nal_off, U);
    r |= dmalloc(&h->d_total, 1);
    r |= dmalloc(&h->d_frame_bytes, F);
    r |= alloc_entropy_buffers(h);
    if (r)
        return r;
    h->eb.hdr_bits = h->d_hdr_bits;
    h->eb.hdr_nbits = h->d_hdr_nbits;
    CK(cudaMemset(h->eb.error, 0, sizeof(int)));
    {
        std::vector<uint32_t> tabs(me_table_words(g.R, me_strip(g.R)));
        me_build_tables(g.R, me_strip(g.R), g.lambda, tabs.data());
        CK(cudaMemcpy(h->d_me_tabs, tabs.data(), tabs.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    }
    CK(cudaMemset(h->d_counters, 0, sizeof(unsigned long long) * (8 + 512)));
    CK(cudaMemset(h->d_mbi[0], 0, sizeof(MbInfo) * g.nmb * L));
    CK(cudaMemset(h->d_mbi[1], 0, sizeof(MbInfo) * g.nmb * L));
    CK(cudaMemset(h->d_rec[0], 0, g.frame_bytes * L));
    CK(cudaMemset(h->d_rec[1], 0, g.frame_bytes * L));
    return 0;
}

void free_buffers(cedar_b200_handle *h)
{
    void *dev[] = {h->d_counters, h->d_raw, h->d_src[0], h->d_src[1], h->d_unf, h->d_rec[0], h->d_rec[1], h->d_mbi[0], h->d_mbi[1],
                   h->d_nnz[0], h->d_nnz[1], h->d_i4[0], h->d_i4[1], h->d_coef[0], h->d_coef[1], h->d_flags, h->d_me_tabs, h->d_pwant, h->d_pcount, h->d_bs,
                   h->d_sse, h->eb.mb_size, h->eb.mb_off, h->d_hdr_bits, h->d_hdr_nbits, h->eb.rbsp_len,
                   h->eb.bins_cursor, h->eb.bins_off, h->eb.bins_len, h->eb.error,
                   h->d_nal_bytes, h->d_nal_off, h->d_total, h->d_frame_bytes};
    free_entropy_buffers(h);
    for (void *p : dev)
        if (p)
            cudaFree(p);
    void *host[] = {h->h_in_luma, h->h_in_chroma, h->h_bytestream, h->h_frame_bytes, h->h_total, h->h_sse,
                    h->h_error, h->h_clip_in};
    for (void *p : host)
        if (p)
            cudaFreeHost(p);
}

// One lock-step pass over s.nlanes lanes (one frame per lane).  t = position inside the GOP (0 => IDR).
//   stream_pre : ingest(t)                                   -> src[p]                 (p = step parity)
//   stream     : intra | ME, residual, MVP/skip; bS; deblock -> syntax[p], unf, rec[t & 1]
//   stream_post: entropy sizes / scan / scatter (as soon as bS / MVP are done, beside the deblocking wavefront), SSE
//                                                            -> RBSP (CAVLC) or bins (CABAC)
//   side stream: cabac_resolve_kernel, cabac_code_kernel
// Buffers with index p are reused two steps later, hence the waits on ev_post[p].
static bool no_overlap_env()
{
    static const bool v = getenv("CEDAR_B200_NO_OVERLAP") != nullptr;
    return v;
}

int encode_step(cedar_b200_handle *h, const Step &s, int t, int gop_pos0, int step_index, bool wait_upload)
{
    const Geom &g = h->g;
    const int nl = s.nlanes, cur = t & 1, frame_i = t == 0, p = step_index & 1;
    const size_t flag_n = (size_t)h->L * g.mbh;
    int *fl_intra = h->d_flags, *fl_y = h->d_flags + flag_n, *fl_c = h->d_flags + 2 * flag_n;
    uint8_t *src = h->d_src[p], *unf = h->d_unf, *rec = h->d_rec[cur], *ref = h->d_rec[cur ^ 1];
    MbInfo *mbi = h->d_mbi[p];
    uint8_t *nnz = h->d_nnz[p], *bs = h->d_bs;
    int16_t *coef = h->d_coef[p];
    const bool no_overlap = no_overlap_env() || h->serialize; // diagnosis / per-kernel timing: everything in line
    cudaStream_t st = h->stream, pre = no_overlap ? st : h->stream_pre, post = no_overlap ? st : h->stream_post;

    // ---- one step ahead: ingest ----
    if (h->post_valid[p])
        CK(cudaStreamWaitEvent(pre, h->ev_post[p], 0)); // step - 2 has finished with src[p] (and main with it)
    if (wait_upload)
        CK(cudaStreamWaitEvent(pre, h->ev_upload[h->upload_deferred_n ? step_index : t], 0));
    LAUNCH_ON(pre, K_INGEST, ingest_kernel, dim3((unsigned)((g.W / 16 + 127) / 128), (unsigned)(g.H + 2 * g.CH), nl), 128, 0, g, s, h->d_raw,
              h->raw_frame_bytes, src);
    CK(cudaEventRecord(h->ev_ingest[p], pre));

    // ---- critical chain ----
    CK(cudaStreamWaitEvent(st, h->ev_ingest[p], 0));
    if (h->post_valid[p])
        CK(cudaStreamWaitEvent(st, h->ev_post[p], 0)); // step - 2 has finished with syntax[p] and rec[cur]
    if (t == 0 && h->post_valid[p ^ 1]) // a new wave of GOPs restarts the rec[] parity: also wait for step - 1's SSE
        CK(cudaStreamWaitEvent(st, h->ev_post[p ^ 1], 0));
    CK(cudaMemsetAsync(h->d_flags, 0, sizeof(int) * 3 * flag_n, st));
    if (frame_i) {
        LAUNCH_ON(st, K_INTRA, intra_kernel, dim3((g.mbh + INTRA_ROWS - 1) / INTRA_ROWS, nl), INTRA_ROWS * 32, 0, g, s, src, unf,
                  mbi, nnz, coef, fl_intra, h->d_i4[p], nullptr, nullptr);
    } else {
        MeShape ms = me_shape(g.R);
        ms.noprune = h->no_prune;
        if (h->count && h->no_prune) // the measurement without pruning: no bound either
            ms.bound = 0;
        ms.exec_count = h->count ? h->d_counters : nullptr;
        const dim3 me_grid((g.mbw + ms.nstrip - 1) / ms.nstrip, (g.mbh + ms.nrow - 1) / ms.nrow, nl);
        const size_t me_smem = me_smem_bytes(g.R, ms.nstrip);
        // the 1080p (R = 16) and 4K (R = 64) geometries have compiled-in row strides
#define ME_LAUNCH(RSW_, COUNT_)                                                                                          \
    LAUNCH_ON(st, K_ME, (me_kernel<RSW_, COUNT_>), me_grid, ME_THREADS, me_smem, g, s, ms, src, ref, mbi, h->d_mbi[p ^ 1], h->d_me_tabs)
        if (h->count) { // the measurement build (executed-instruction counter, CEDAR_B200_NO_PRUNE)
            switch (ms.RSW) {
            case 27: ME_LAUNCH(27, true); break;
            case 43: ME_LAUNCH(43, true); break;
            default: ME_LAUNCH(0, true); break;
            }
        } else {
            switch (ms.RSW) {
            case 27: ME_LAUNCH(27, false); break;
            case 43: ME_LAUNCH(43, false); break;
            default: ME_LAUNCH(0, false); break;
            }
        }
#undef ME_LAUNCH
        LAUNCH_ON(st, K_INTER, inter_kernel, dim3((g.nmb + 3) / 4, nl), 128, 0, g, s, src, ref, unf, mbi, nnz, coef);
        if (g.p_intra) { // decide (parallel), then re-code the chosen macroblocks as intra in wavefront order
            CK(cudaMemsetAsync(h->d_pcount, 0, sizeof(int) * h->L, st));
            LAUNCH_ON(st, K_PINTRA, pintra_decide_kernel, dim3((g.nmb + 3) / 4, nl), 128, 0, g, s, src, unf, mbi, h->d_pwant,
                      h->d_pcount);
            LAUNCH_ON(st, K_INTRA, intra_kernel, dim3((g.mbh + INTRA_ROWS - 1) / INTRA_ROWS, nl), INTRA_ROWS * 32, 0, g, s, src, unf,
                      mbi, nnz, coef, fl_intra, h->d_i4[p], h->d_pwant, h->d_pcount);
        }
    }
    // boundary strengths; on inter steps the same launch runs median MV prediction / the skip decision (K2)
    LAUNCH_ON(st, K_BS, bs_kernel, dim3((g.nmb * 8 + 127) / 128, nl), 128, 0, g, s, mbi, nnz, bs, !frame_i);
    CK(cudaEventRecord(h->ev_syn[p], st)); // the syntax records are final: entropy coding does not wait for deblocking
    // equally tall CTAs of at most DB_ROWS macroblock rows (1080p: 4 x 17, 720p: 3 x 15, 4K: 8 x 17)
    const int db_ctas = (g.mbh + DB_ROWS - 1) / DB_ROWS, db_rows = (g.mbh + db_ctas - 1) / db_ctas;
    LAUNCH_ON(st, K_DEBLOCK, deblock_kernel, dim3((g.mbh + db_rows - 1) / db_rows, nl, 2), (db_rows + 2) * 32, 0, g, s, unf,
              rec, bs, fl_y, fl_c, db_rows);
    CK(cudaEventRecord(h->ev_main[p], st));

    // ---- beside and behind the chain: the parallel entropy passes (from the syntax records, while the wavefront of
    // deblock_kernel runs), then the statistics of the deblocked picture ----
    CK(cudaStreamWaitEvent(post, h->ev_syn[p], 0));
    dim3 egrid((g.nmb + g.nslices + 127) / 128, nl);
    EntropyBufs eb = h->eb;
    eb.i4 = h->d_i4[p];
    LAUNCH_ON(post, K_ESIZE, entropy_size_kernel, egrid, 128, 0, g, s, frame_i, mbi, nnz, coef, eb);
    LAUNCH_ON(post, K_ESCAN, entropy_scan_kernel, dim3(1, nl), 1024, 0, g, s, h->eb);
    if (!g.cabac)
        LAUNCH_ON(post, K_EZERO, rbsp_zero_kernel, dim3(8, nl, g.nslices), 256, 0, s, h->eb.rbsp, h->eb.rbsp_cap,
                  h->eb.rbsp_len);
    LAUNCH_ON(post, K_EWRITE, entropy_write_kernel, egrid, 128, 0, g, s, frame_i, mbi, nnz, coef, eb);
    CK(cudaEventRecord(h->ev_ent[p], post));
    CK(cudaStreamWaitEvent(post, h->ev_main[p], 0));
    LAUNCH_ON(post, K_SSE, sse_kernel, dim3(32, nl), 256, 0, g, s, src, rec, h->d_sse);
    CK(cudaEventRecord(h->ev_post[p], post));
    h->post_valid[p] = true;
    if (g.cabac) {
        // the bins of these frames are final: code them on a side stream while the next frames are reconstructed
        cudaStream_t side = no_overlap ? st : h->stream_cabac[h->side_next];
        CK(cudaStreamWaitEvent(side, h->ev_ent[p], 0));
        LAUNCH_ON(side, K_CRESOLVE, cabac_resolve_kernel, nl * g.nslices, RES_THREADS, RES_SMEM_BYTES, g, s, h->K, gop_pos0, h->eb,
                  h->count ? h->d_counters + 8 : nullptr);
        EntropyBufs ebc = h->eb; // the limb scratch of this side stream (its launches are serialised)
        ebc.limbs += (size_t)(no_overlap || !h->clip_mode ? 0 : h->side_next) * h->L * g.nslices * h->eb.limb_cap;
        LAUNCH_ON(side, K_CCODE, cabac_code_kernel, nl * g.nslices, CP_THREADS, CP_SMEM_BYTES, g, s, ebc);
        if (!no_overlap) {
            h->side_used |= 1u << h->side_next;
            h->side_next = (h->side_next + 1) % cedar_b200_handle::NSIDE;
        }
    }
    h->last_cur = cur;
    h->last_par = p;
    return 0;
}

// Serial CABAC stage (all frames at once), emulation prevention and packing of `nframes` frames.
int finish_stream(cedar_b200_handle *h, int nframes, int gop_pos0, bool with_param_sets)
{
    CK(cudaEventRecord(h->ev_post_done, h->stream_post));
    CK(cudaStreamWaitEvent(h->stream, h->ev_post_done, 0));
    for (int i = 0; i < cedar_b200_handle::NSIDE; i++)
        if (h->side_used & (1u << i)) {
            CK(cudaEventRecord(h->ev_cabac[i], h->stream_cabac[i]));
            CK(cudaStreamWaitEvent(h->stream, h->ev_cabac[i], 0));
        }
    h->side_used = 0;
    unsigned cpf = h->chunks_per_frame;
    const int nunits = nframes * h->S; // slice NALs
    const unsigned cblocks = (cpf + 255) / 256; // grid.x = units x chunk blocks (gridDim.y would cap the units at 65535)
    LAUNCH(K_EPBCOUNT, epb_count_kernel, (unsigned)nunits * cblocks, 256, 0, nunits, h->eb.rbsp, h->eb.rbsp_cap,
           h->eb.rbsp_len, h->d_chunk_cnt, cpf, cblocks);
    ParamSets ps;
    memset(&ps, 0, sizeof(ps));
    memcpy(ps.bytes, h->prefix, (size_t)h->prefix_len);
    ps.len = h->prefix_len;
    ps.mode = h->cfg.repeat_headers ? 2 : (with_param_sets ? 1 : 0); // cedar.c:1058-1061: once, before stream frame 0
    LAUNCH(K_EPBSCAN, epb_scan_kernel, nunits, 1024, 0, nunits, h->eb.rbsp_len, h->d_chunk_cnt, cpf, h->d_nal_bytes, ps, h->S,
           h->K, gop_pos0);
    LAUNCH(K_PACKSCAN, pack_scan_kernel, 1, 1024, 0, nunits, h->S, h->d_nal_bytes, 0u, h->d_nal_off, h->d_frame_bytes,
           h->d_total, (unsigned long long)h->out_cap, h->eb.error);
    LAUNCH(K_EPBWRITE, epb_write_kernel, (unsigned)nunits * cblocks, 256, 0, nunits, h->S, h->K, gop_pos0, h->eb.rbsp,
           h->eb.rbsp_cap, h->eb.rbsp_len, h->d_chunk_cnt, cpf, cblocks, h->d_nal_off, h->d_total, h->d_out, ps);
    return 0;
}

// Slice-header bits of every unit a clip (or a frame-mode call) can address, written once at open(): the bits depend
// only on the frame's position in its GOP and on the slice (cedar.c:984-1030: slice type, frame_num = frame_p_count & 15),
// clips start at a GOP boundary, so entry (f, k) serves frame f of any clip, and frame mode points the entropy passes at
// the row of its current frame_p_count.
int build_header_table(cedar_b200_handle *h)
{
    const int S = h->S, rows = h->F > h->K ? h->F : h->K;
    std::vector<unsigned long long> bits((size_t)rows * S);
    std::vector<int> nbits((size_t)rows * S);
    for (int f = 0; f < rows; f++) {
        int p = f % h->K;
        for (int k = 0; k < S; k++) { // first_mb_in_slice = first macroblock of the slice's first row (0: cedar.c:992-993)
            uint64_t b = 0;
            int r = cedar_hdr_slice_mb(p == 0, p, h->g.cabac, k * h->g.srows * h->g.mbw, &b, &nbits[(size_t)f * S + k]);
            if (r)
                return r;
            bits[(size_t)f * S + k] = b;
        }
    }
    CK(cudaMemcpy(h->d_hdr_bits, bits.data(), sizeof(unsigned long long) * bits.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->d_hdr_nbits, nbits.data(), sizeof(int) * nbits.size(), cudaMemcpyHostToDevice));
    return 0;
}

int begin_stream(cedar_b200_handle *h, int nframes)
{
    CK(cudaMemsetAsync(h->eb.bins_cursor, 0, sizeof(unsigned long long), h->stream));
    CK(cudaMemsetAsync(h->d_sse, 0, sizeof(unsigned long long) * nframes, h->stream));
    CK(cudaMemsetAsync(h->eb.rbsp_len, 0, sizeof(uint32_t) * nframes * h->S, h->stream));
    CK(cudaMemsetAsync(h->eb.bins_len, 0, sizeof(uint32_t) * nframes * h->S, h->stream));
    CK(cudaEventRecord(h->ev_begin, h->stream));
    CK(cudaStreamWaitEvent(h->stream_pre, h->ev_begin, 0));
    CK(cudaStreamWaitEvent(h->stream_post, h->ev_begin, 0));
    h->post_valid[0] = h->post_valid[1] = false;
    return 0;
}

int check_error(cedar_b200_handle *h)
{
    if (*h->h_error) {
        fprintf(stderr, "cedar_b200: device buffer overflow (code %d): bitstream larger than the configured bound.\n",
                *h->h_error);
        cudaMemset(h->eb.error, 0, sizeof(int));
        return -ENOMEM;
    }
    return 0;
}

} // namespace

extern "C" {

const char *cedar_b200_version(void) { return "cedar_b200 0.1 (sm_100a)"; }

int cedar_b200_write_sps(const struct cedar_b200_config *cfg, uint8_t *out, int cap)
{
    const int wmb = (int)ALIGN_UP(cfg->dst_width, 16) >> 4, hmb = (int)ALIGN_UP(cfg->dst_height, 16) >> 4;
    return cedar_hdr_sps(cfg->profile, cfg->auto_level ? cedar_hdr_min_level(wmb * hmb) : cfg->level, wmb, hmb,
                         cfg->sps_crop ? (wmb * 16 - cfg->src_width) / 2 : 0,
                         cfg->sps_crop ? (hmb * 16 - cfg->src_height) / 2 : 0, out, cap);
}
int cedar_b200_write_pps(const struct cedar_b200_config *cfg, uint8_t *out, int cap)
{
    return cedar_hdr_pps(cfg->qp, cfg->entropy_coding_mode == CEDAR_B200_ENTROPY_CABAC, out, cap);
}
int cedar_b200_slice_header(int frame_i, int frame_p_count, int cabac, uint32_t *bits, int *nbits)
{
    return cedar_hdr_slice(frame_i, frame_p_count, cabac, bits, nbits);
}
int cedar_b200_slice_header_mb(int frame_i, int frame_p_count, int cabac, int first_mb, uint64_t *bits, int *nbits)
{
    return cedar_hdr_slice_mb(frame_i, frame_p_count, cabac, first_mb, bits, nbits);
}

// Everything a handle owns, in the order cedar_b200_close releases it; also the unwinding of a failed open()
// (members are zero until they are created: the handle is value-initialised).
static void destroy_handle(cedar_b200_handle *h)
{
    const auto t0 = std::chrono::steady_clock::now();
    const bool trace = getenv("CEDAR_B200_TRACE") != nullptr && !h->pipe;
    if (h->pipe)
        cedar_b200_pipe_close(h->pipe);
    for (cudaEvent_t e : h->ev_pool)
        cudaEventDestroy(e);
    free_buffers(h);
    cudaEvent_t evs[] = {h->ev_begin, h->ev_post_done, h->ev_encode_done, h->ev_ingest[0], h->ev_ingest[1],
                         h->ev_main[0], h->ev_main[1], h->ev_post[0], h->ev_post[1], h->ev_syn[0], h->ev_syn[1], h->ev_ent[0],
                         h->ev_ent[1]};
    for (cudaEvent_t e : evs)
        if (e)
            cudaEventDestroy(e);
    for (auto &e : h->ev_upload)
        if (e)
            cudaEventDestroy(e);
    for (int i = 0; i < cedar_b200_handle::NSIDE; i++) {
        if (h->ev_cabac[i])
            cudaEventDestroy(h->ev_cabac[i]);
        if (h->stream_cabac[i])
            cudaStreamDestroy(h->stream_cabac[i]);
    }
    cudaStream_t sts[] = {h->stream_copy, h->stream_pre, h->stream_post, h->stream};
    for (cudaStream_t st : sts)
        if (st)
            cudaStreamDestroy(st);
    delete h;
    if (trace)
        fprintf(stderr, "[trace] close: buffers, streams and events released in %.1f ms\n",
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
}

// Queued mode (cfg.queue_gops): the handle is a front over a pipeline of worker handles (pipeline.cpp).
static int open_queued(const struct cedar_b200_config *cfg, struct cedar_b200_io *io, cedar_b200_handle *h)
{
    cedar_b200_config wc = *cfg;
    wc.queue_gops = 0;
    int r = cedar_b200_pipe_open(&wc, nullptr, 0, 2, cfg->queue_gops, &h->pipe);
    if (r)
        return r;
    const Geom &g = h->g;
    h->in_luma_size = (int)ALIGN_UP((size_t)g.src_w * g.src_h, 4096);
    size_t chroma_bytes = (size_t)g.src_w * g.src_h / (g.src_format == CEDAR_B200_FORMAT_NV16 ? 1 : 2);
    h->in_chroma_size = (int)ALIGN_UP(chroma_bytes, 4096);
    h->bytestream_size = (int)ALIGN_UP((size_t)g.nmb * 1536 + 4096, 4096);
    r |= hmalloc(&h->h_in_luma, h->in_luma_size);
    r |= hmalloc(&h->h_in_chroma, h->in_chroma_size);
    r |= hmalloc(&h->h_bytestream, h->bytestream_size);
    r |= hmalloc(&h->h_sse, 1);
    if (r)
        return r;
    h->q_cap = cfg->queue_gops * h->K;
    io->input_luma = h->h_in_luma;
    io->input_luma_size = h->in_luma_size;
    io->input_chroma = h->h_in_chroma;
    io->input_chroma_size = h->in_chroma_size;
    io->bytestream = h->h_bytestream;
    io->bytestream_size = h->bytestream_size;
    return 0;
}

int cedar_b200_open(const struct cedar_b200_config *cfg, struct cedar_b200_io *io, cedar_b200_handle **out)
{
    if (!cfg || !io || !out)
        return -EINVAL;
    int r = validate(cfg);
    if (r)
        return r;
    // The serial CABAC stages of successive steps run concurrently on side streams; with the default of 8 hardware
    // connections streams share queues and serialise.  CUDA_DEVICE_MAX_CONNECTIONS=32 must be in the environment before
    // CUDA initialises in the host process: the CLI and bench.py export it themselves; a library does not touch its
    // host's environment (INTEGRATION.md 4).
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || cfg->device >= ndev || cfg->device < 0) {
        fprintf(stderr, "cedar_b200: no usable CUDA device (this encoder has no CPU fallback).\n");
        return -ENODEV;
    }
    if (cudaSetDevice(cfg->device) != cudaSuccess)
        return -ENODEV;
    cedar_b200_handle *h = new cedar_b200_handle();
    h->cfg = *cfg;
    h->device = cfg->device;
    h->t_open = std::chrono::steady_clock::now();
    Geom &g = h->g;
    g.W = cfg->dst_width;
    g.H = cfg->dst_height;
    g.CW = g.W / 2;
    g.CH = g.H / 2;
    g.mbw = g.W >> 4;
    g.mbh = g.H >> 4;
    g.nmb = g.mbw * g.mbh;
    g.src_w = cfg->src_width;
    g.src_h = cfg->src_height;
    g.src_format = cfg->src_format;
    g.qp = cfg->qp;
    int qpi = cfg->qp + 4; // chroma_qp_index_offset = 4 (cedar.c:969-971, PARA1 cedar.c:1165-1168)
    g.qpc = kChromaQp[qpi < 0 ? 0 : (qpi > 51 ? 51 : qpi)];
    g.R = cfg->me_range ? cfg->me_range : 16;
    int lq = (cfg->qp - 12) / 6;
    g.lambda = 1 << (lq < 0 ? 0 : (lq > 5 ? 5 : lq));
    g.cabac = cfg->entropy_coding_mode == CEDAR_B200_ENTROPY_CABAC;
    g.srows = cfg->slice_rows > 0 && cfg->slice_rows < g.mbh ? cfg->slice_rows : g.mbh;
    g.nslices = (g.mbh + g.srows - 1) / g.srows;
    g.intra4x4 = cfg->intra4x4 != 0;
    g.p_intra = cfg->p_intra != 0;
    h->S = g.nslices;
    g.frame_bytes = (unsigned long long)g.W * g.H * 3 / 2;
    h->K = cfg->keyframe_interval;
    h->clip_mode = cfg->max_clip_frames > 0;
    h->F = h->clip_mode ? cfg->max_clip_frames : 1;
    h->raw_frame_bytes = (size_t)g.src_w * g.src_h * (g.src_format == CEDAR_B200_FORMAT_NV16 ? 2 : 3) /
                         (g.src_format == CEDAR_B200_FORMAT_NV16 ? 1 : 2);
    h->grow = 1;
    h->no_prune = getenv("CEDAR_B200_NO_PRUNE") != nullptr;
    if (cfg->queue_gops > 0) {
        r = open_queued(cfg, io, h);
        if (r) {
            destroy_handle(h);
            return r;
        }
        *out = h;
        return 0;
    }
    int gops = (h->F + h->K - 1) / h->K;
    int lanes = cfg->gops_in_flight > 0 ? cfg->gops_in_flight : 16;
    if (lanes > gops)
        lanes = gops;
    while (lanes > 1 && (long)lanes * g.mbh > 148L * 16) // keep every wavefront CTA resident
        lanes--;
    if (cfg->gops_in_flight <= 0) { // auto: equal waves (20 GOPs run as 10 + 10, not 16 + 4)
        const int waves = (gops + lanes - 1) / lanes;
        lanes = (gops + waves - 1) / waves;
    }
    h->L = lanes;
    // Stream priorities were measured (main stream high / entropy streams low, and the reverse): within 1.5 % of
    // plain default priorities, which are the fastest (80.1 ms per 1080p clip against 81.4), so none are set.
    auto mkstream = [](cudaStream_t *st) { return cudaStreamCreateWithFlags(st, cudaStreamNonBlocking) == cudaSuccess; };
    auto mkevent = [](cudaEvent_t *e) { return cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess; };
    bool ok = mkstream(&h->stream) && mkstream(&h->stream_pre) && mkstream(&h->stream_post) && mkstream(&h->stream_copy) &&
              mkevent(&h->ev_begin) && mkevent(&h->ev_post_done) && mkevent(&h->ev_encode_done);
    for (int i = 0; ok && i < 2; i++)
        ok = mkevent(&h->ev_ingest[i]) && mkevent(&h->ev_main[i]) && mkevent(&h->ev_post[i]) && mkevent(&h->ev_syn[i]) &&
             mkevent(&h->ev_ent[i]);
    {
        const char *ua = getenv("CEDAR_B200_UPLOAD_AHEAD");
        h->upload_ahead = ua ? atoi(ua) : 1;
        if (h->upload_ahead < 0)
            h->upload_ahead = 0;
        h->upload_deferred_n = 0;
    }
    // one event per pass of the longest clip: K passes per wave of L GOPs
    h->ev_upload.assign(h->clip_mode ? (size_t)h->K * (size_t)(((h->F + h->K - 1) / h->K + h->L - 1) / h->L) : 0, nullptr);
    for (auto &e : h->ev_upload)
        ok = ok && mkevent(&e);
    for (int i = 0; ok && i < cedar_b200_handle::NSIDE; i++)
        ok = mkstream(&h->stream_cabac[i]) && mkevent(&h->ev_cabac[i]);
    if (!ok) {
        fprintf(stderr, "cedar_b200: could not create streams / events: %s\n", cudaGetErrorString(cudaGetLastError()));
        destroy_handle(h);
        return -ENODEV;
    }
    if (cudaFuncSetAttribute(cabac_code_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CP_SMEM_BYTES) != cudaSuccess ||
        cudaFuncSetAttribute(cabac_resolve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, RES_SMEM_BYTES) != cudaSuccess) {
        fprintf(stderr, "cedar_b200: the CABAC kernels need %d / %d bytes of shared memory\n", CP_SMEM_BYTES, RES_SMEM_BYTES);
        cudaGetLastError();
        destroy_handle(h);
        return -ENODEV;
    }
    const int me_smem = (int)me_smem_bytes(g.R, me_strip(g.R));
    if (cudaFuncSetAttribute(me_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, me_smem) != cudaSuccess ||
        cudaFuncSetAttribute(me_kernel<27>, cudaFuncAttributeMaxDynamicSharedMemorySize, me_smem) != cudaSuccess ||
        cudaFuncSetAttribute(me_kernel<43>, cudaFuncAttributeMaxDynamicSharedMemorySize, me_smem) != cudaSuccess ||
        cudaFuncSetAttribute(me_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, me_smem) != cudaSuccess ||
        cudaFuncSetAttribute(me_kernel<27, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, me_smem) != cudaSuccess ||
        cudaFuncSetAttribute(me_kernel<43, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, me_smem) != cudaSuccess) {
        fprintf(stderr, "cedar_b200: search range %d needs more shared memory than the device offers\n", g.R);
        cudaGetLastError();
        destroy_handle(h);
        return -EINVAL;
    }
    const auto t_alloc = std::chrono::steady_clock::now();
    r = alloc_buffers(h);
    if (!r)
        r = build_header_table(h);
    if (getenv("CEDAR_B200_TRACE"))
        fprintf(stderr, "[trace] open: context + streams %.1f ms, buffers %.1f ms (clip capacity %d frames, %d GOPs in flight)\n",
                std::chrono::duration<double, std::milli>(t_alloc - h->t_open).count(),
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_alloc).count(), h->F, h->L);
    // SPS + PPS, emitted once before the first frame (cedar.c:1058-1061)
    int n1 = r ? 0 : cedar_b200_write_sps(cfg, h->prefix, 40);
    int n2 = r || n1 < 0 ? 0 : cedar_b200_write_pps(cfg, h->prefix + n1, 24);
    if (!r && (n1 < 0 || n2 < 0))
        r = -EINVAL;
    if (r) {
        destroy_handle(h);
        return r;
    }
    h->prefix_len = n1 + n2;
    io->input_luma = h->h_in_luma;
    io->input_luma_size = h->in_luma_size;
    io->input_chroma = h->h_in_chroma;
    io->input_chroma_size = h->in_chroma_size;
    io->bytestream = h->h_bytestream;
    io->bytestream_size = h->bytestream_size;
    *out = h;
    return 0;
}

// Queued mode: frame t goes into the batch being filled; a full batch is handed to the pipeline (asynchronous); the call
// returns the bytes of frame t - 2 * batch (0 before that): while batch j fills, batch j - 1 is being encoded and batch
// j - 2 is handed out, so the producer never waits unless the GPU is the slower side.
static int queued_take_frame(cedar_b200_handle *h)
{
    if (h->q_pos >= h->q_sizes.size()) { // next finished batch, copied out so that its worker is free again at once
        const uint8_t *out = nullptr;
        const int *sizes = nullptr;
        const double *sse = nullptr;
        int n = 0;
        long long total = cedar_b200_pipe_next(h->pipe, &out, &sizes, &n, &sse, 1);
        if (total <= 0)
            return (int)total;
        h->q_bytes.assign(out, out + total);
        h->q_sizes.assign(sizes, sizes + n);
        h->q_sse.assign(sse, sse + n);
        h->q_pos = 0, h->q_off = 0;
        cedar_b200_pipe_release(h->pipe);
    }
    const int sz = h->q_sizes[h->q_pos];
    if (sz > h->bytestream_size)
        return -ENOMEM;
    memcpy(h->h_bytestream, h->q_bytes.data() + h->q_off, (size_t)sz);
    h->h_sse[0] = (unsigned long long)h->q_sse[h->q_pos]; // cedar_b200_stats: the frame just handed out
    h->last_nframes = 1;
    h->sse_valid = true;
    h->q_off += (size_t)sz;
    h->q_pos++;
    h->q_out++;
    return sz;
}

static int queued_encode_frame(cedar_b200_handle *h)
{
    const size_t luma_bytes = (size_t)h->g.src_w * h->g.src_h;
    int ret = 0;
    if (h->q_in >= 2LL * h->q_cap) { // before the slot of batch j is acquired: batch j - 2 frees its worker
        ret = queued_take_frame(h);
        if (ret < 0)
            return ret;
    }
    if (!h->q_staging) {
        int cap = 0;
        h->q_staging = (uint8_t *)cedar_b200_pipe_acquire(h->pipe, &h->q_frame_bytes, &cap);
        if (!h->q_staging || cap != h->q_cap || h->q_frame_bytes != h->raw_frame_bytes)
            return -EIO;
        h->q_fill = 0;
    }
    uint8_t *dst = h->q_staging + (size_t)h->q_fill * h->q_frame_bytes;
    memcpy(dst, h->h_in_luma, luma_bytes);
    memcpy(dst + luma_bytes, h->h_in_chroma, h->raw_frame_bytes - luma_bytes);
    h->q_in++;
    if (++h->q_fill == h->q_cap) {
        int r = cedar_b200_pipe_submit(h->pipe, h->q_fill);
        h->q_staging = nullptr;
        if (r)
            return r;
    }
    // cedar.c:1193-1196
    h->frame_p_count++;
    if (h->frame_p_count == h->K)
        h->frame_p_count = 0;
    h->frame_count++;
    return ret;
}

int cedar_b200_flush(cedar_b200_handle *h)
{
    if (!h)
        return -EINVAL;
    if (!h->pipe)
        return 0;
    auto t0 = std::chrono::steady_clock::now();
    if (h->q_staging) { // the partial last batch
        int r = cedar_b200_pipe_submit(h->pipe, h->q_fill);
        h->q_staging = nullptr;
        if (r)
            return r;
    }
    cedar_b200_pipe_finish(h->pipe);
    int ret = h->q_out < h->q_in ? queued_take_frame(h) : 0;
    h->busy_ns += std::chrono::duration<double, std::nano>(std::chrono::steady_clock::now() - t0).count();
    return ret;
}

int cedar_b200_encode_frame(cedar_b200_handle *h)
{
    if (!h)
        return -EINVAL; // cedar.c:1039-1043: not configured
    if (h->pipe) {
        auto tq = std::chrono::steady_clock::now();
        int rq = queued_encode_frame(h);
        h->busy_ns += std::chrono::duration<double, std::nano>(std::chrono::steady_clock::now() - tq).count();
        return rq;
    }
    cudaSetDevice(h->device);
    auto t0 = std::chrono::steady_clock::now();
    const Geom &g = h->g;
    size_t luma_bytes = (size_t)g.src_w * g.src_h;
    CK(cudaMemcpyAsync(h->d_raw, h->h_in_luma, luma_bytes, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_raw + luma_bytes, h->h_in_chroma, h->raw_frame_bytes - luma_bytes, cudaMemcpyHostToDevice,
                       h->stream));
    int r;
    h->eb.hdr_bits = h->d_hdr_bits + (size_t)h->frame_p_count * h->S; // the header row of this GOP position
    h->eb.hdr_nbits = h->d_hdr_nbits + (size_t)h->frame_p_count * h->S;
    if ((r = begin_stream(h, 1)))
        return r;
    Step s = {1, 0, 1, 1};
    if ((r = encode_step(h, s, h->frame_p_count, h->frame_p_count, 0, false)))
        return r;
    if ((r = finish_stream(h, 1, h->frame_p_count, h->frame_count == 0)))
        return r;
    CK(cudaMemcpyAsync(h->h_total, h->d_total, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(h->h_error, h->eb.error, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(h->h_sse, h->d_sse, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if ((r = check_error(h)))
        return r;
    size_t total = (size_t)*h->h_total;
    if (total == 0 || total > (size_t)h->bytestream_size)
        return -ENOMEM;
    CK(cudaMemcpyAsync(h->h_bytestream, h->d_out, total, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->last_nframes = 1;
    h->sse_valid = true;
    // cedar.c:1193-1196 (the reference swap of :1198-1201 is the `t & 1` buffer choice in encode_step)
    h->frame_p_count++;
    if (h->frame_p_count == h->K)
        h->frame_p_count = 0;
    h->frame_count++;
    h->busy_ns += std::chrono::duration<double, std::nano>(std::chrono::steady_clock::now() - t0).count();
    return (int)total;
}

void *cedar_b200_clip_input(cedar_b200_handle *h, size_t *frame_bytes)
{
    if (!h)
        return nullptr;
    if (frame_bytes)
        *frame_bytes = h->raw_frame_bytes;
    return h->h_clip_in;
}

int cedar_b200_clip_upload(cedar_b200_handle *h, int nframes)
{
    if (!h || !h->h_clip_in || nframes <= 0 || nframes > h->F)
        return -EINVAL;
    cudaSetDevice(h->device);
    if (h->upload_ahead > 0) { // paced: the copies are issued by the clip_encode that follows (upload_pass)
        h->upload_deferred_n = nframes;
        h->upload_pending = true;
        return 0;
    }
    h->upload_deferred_n = 0;
    // Copies are issued in the order the encoder consumes the frames (step t needs frame t of every GOP) on a
    // dedicated stream; clip_encode's step t waits for ev_upload[t] only, so the transfer overlaps the encode.
    CK(cudaEventRecord(h->ev_encode_done, h->stream)); // do not overwrite frames a running encode still reads
    CK(cudaStreamWaitEvent(h->stream_copy, h->ev_encode_done, 0));
    const int K = h->K, gops = (nframes + K - 1) / K;
    const size_t fb = h->raw_frame_bytes;
    for (int t = 0; t < K; t++) {
        for (int gp = 0; gp < gops; gp++) {
            size_t f = (size_t)gp * K + t;
            if (f < (size_t)nframes)
                CK(cudaMemcpyAsync(h->d_raw + f * fb, h->h_clip_in + f * fb, fb, cudaMemcpyHostToDevice, h->stream_copy));
        }
        CK(cudaEventRecord(h->ev_upload[t], h->stream_copy));
    }
    h->upload_pending = true;
    return 0;
}

// Paced upload: the host -> device copies of pass j (frame t = j % K of the GOPs of wave j / K) on the copy stream, behind
// `gate` (an event of the pass `upload_ahead` passes earlier); ev_upload[j] tells the pass that its frames are resident.
static int upload_pass(cedar_b200_handle *h, int nframes, int j, cudaEvent_t gate)
{
    const int K = h->K, gops = (nframes + K - 1) / K, t = j % K, gop0 = (j / K) * h->L;
    if (j >= (int)h->ev_upload.size() || gop0 >= gops)
        return 0;
    const size_t fb = h->raw_frame_bytes;
    CK(cudaStreamWaitEvent(h->stream_copy, gate, 0));
    for (int gp = gop0; gp < gops && gp < gop0 + h->L; gp++) {
        const size_t f = (size_t)gp * K + t;
        if (f < (size_t)nframes)
            CK(cudaMemcpyAsync(h->d_raw + f * fb, h->h_clip_in + f * fb, fb, cudaMemcpyHostToDevice, h->stream_copy));
    }
    CK(cudaEventRecord(h->ev_upload[j], h->stream_copy));
    return 0;
}

// Issues the whole encode of the clip that is resident in d_raw (asynchronous).
static int run_clip(cedar_b200_handle *h, int nframes, int first_frame_index)
{
    int r;
    h->eb.hdr_bits = h->d_hdr_bits;
    h->eb.hdr_nbits = h->d_hdr_nbits;
    if ((r = begin_stream(h, nframes)))
        return r;
    const int K = h->K, gops = (nframes + K - 1) / K;
    const bool paced = h->upload_pending && h->upload_deferred_n > 0;
    const int up_n = h->upload_deferred_n, D = h->upload_ahead;
    if (paced) {
        // the first D passes: as soon as no earlier ingest reads d_raw any more (all of them are on stream_pre)
        CK(cudaEventRecord(h->ev_encode_done, (h->serialize || no_overlap_env()) ? h->stream : h->stream_pre));
        for (int j = 0; j < D; j++)
            if ((r = upload_pass(h, up_n, j, h->ev_encode_done)))
                return r;
    }
    int step_index = 0;
    for (int gop0 = 0; gop0 < gops; gop0 += h->L) {
        int nl = gops - gop0 < h->L ? gops - gop0 : h->L;
        for (int t = 0; t < K; t++) {
            Step s = {nl, gop0 * K + t, K, nframes};
            if (s.frame0 >= nframes)
                break;
            if (paced && step_index != (gop0 / h->L) * K + t)
                return -EIO; // pass numbering of upload_pass and of this loop must agree
            if ((r = encode_step(h, s, t, 0, step_index, h->upload_pending)))
                return r;
            if (paced && (r = upload_pass(h, up_n, step_index + D, h->ev_ingest[step_index & 1])))
                return r;
            step_index++;
        }
    }
    if (paced && up_n > nframes) { // a clip_upload of more frames than this encode covers: the rest of it now, and
                                   // every later ingest behind it (nothing else would wait for these copies)
        const int last = (int)h->ev_upload.size() - 1;
        for (int j = step_index + D; j <= last; j++)
            if ((r = upload_pass(h, up_n, j, h->ev_ingest[(step_index - 1) & 1])))
                return r;
        CK(cudaEventRecord(h->ev_upload[last], h->stream_copy));
        CK(cudaStreamWaitEvent((h->serialize || no_overlap_env()) ? h->stream : h->stream_pre, h->ev_upload[last], 0));
    }
    h->upload_pending = false;
    h->upload_deferred_n = 0;
    return finish_stream(h, nframes, 0, first_frame_index == 0);
}

int cedar_b200_clip_encode(cedar_b200_handle *h, int nframes, int first_frame_index)
{
    if (!h || !h->clip_mode || nframes <= 0 || nframes > h->F || first_frame_index < 0 || (first_frame_index % h->K) != 0)
        return -EINVAL;
    cudaSetDevice(h->device);
    auto t0 = std::chrono::steady_clock::now();
    int r = run_clip(h, nframes, first_frame_index);
    if (r)
        return r;
    h->last_nframes = nframes;
    h->sse_valid = false;
    h->last_first_frame = first_frame_index;
    h->busy_ns += std::chrono::duration<double, std::nano>(std::chrono::steady_clock::now() - t0).count();
    return 0;
}

long long cedar_b200_clip_download(cedar_b200_handle *h, const uint8_t **out, int *frame_bytes)
{
    if (!h || !h->h_clip_out || h->last_nframes <= 0)
        return -EINVAL;
    cudaSetDevice(h->device);
    int n = h->last_nframes;
    for (;;) {
        CK(cudaMemcpyAsync(h->h_total, h->d_total, sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(h->h_error, h->eb.error, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(h->h_frame_bytes, h->d_frame_bytes, sizeof(int) * n, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(h->h_sse, h->d_sse, sizeof(unsigned long long) * n, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (!*h->h_error)
            break;
        // The coded clip did not fit the heuristic bounds of the entropy buffers (nothing was written out of bounds:
        // every writer checks).  The raw clip is still resident: enlarge the buffers and encode it again.
        if (h->grow >= 256 || getenv("CEDAR_B200_NO_GROW"))
            return check_error(h);
        fprintf(stderr, "cedar_b200: coded clip exceeds the entropy buffer bounds (code %d): enlarging them x4 and encoding again\n",
                *h->h_error);
        CK(cudaMemset(h->eb.error, 0, sizeof(int)));
        CK(cudaDeviceSynchronize());
        h->grow *= 4;
        free_entropy_buffers(h);
        int r = alloc_entropy_buffers(h);
        if (r) { // no memory for the larger buffers: back to the size that worked, and report
            h->grow /= 4;
            free_entropy_buffers(h);
            if (alloc_entropy_buffers(h))
                fprintf(stderr, "cedar_b200: could not restore the entropy buffers; the handle is unusable\n");
            return r;
        }
        if ((r = run_clip(h, n, h->last_first_frame)))
            return r;
    }
    h->sse_valid = true;
    size_t total = (size_t)*h->h_total;
    if (total == 0 || total > h->out_cap)
        return -ENOMEM;
    CK(cudaMemcpyAsync(h->h_clip_out, h->d_out, total, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (out)
        *out = h->h_clip_out;
    if (frame_bytes)
        memcpy(frame_bytes, h->h_frame_bytes, sizeof(int) * n);
    return (long long)total;
}

int cedar_b200_stats(cedar_b200_handle *h, double *sse_y, int nframes)
{
    if (!h || !sse_y || nframes <= 0 || nframes > h->last_nframes)
        return -EINVAL;
    if (!h->sse_valid) { // clip_encode without clip_download so far: fetch the statistics of that encode
        cudaSetDevice(h->device);
        CK(cudaMemcpyAsync(h->h_sse, h->d_sse, sizeof(unsigned long long) * h->last_nframes, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        h->sse_valid = true;
    }
    for (int i = 0; i < nframes; i++)
        sse_y[i] = (double)h->h_sse[i];
    return 0;
}

int cedar_b200_profile_enable(cedar_b200_handle *h, int enable)
{
    if (!h || h->pipe)
        return -EINVAL;
    cudaSetDevice(h->device);
    if (!enable && h->prof)
        prof_collect(h);
    h->prof = enable != 0;
    h->serialize = enable >= 2;
    h->count = enable == 3;
    return 0;
}

int cedar_b200_profile_read(cedar_b200_handle *h, const char **names, float *ms, int *launches, int cap, int reset)
{
    if (!h || h->pipe)
        return -EINVAL;
    cudaSetDevice(h->device);
    prof_collect(h);
    int n = 0;
    for (int i = 0; i < K_COUNT && n < cap; i++) {
        if (!h->prof_n[i])
            continue;
        if (names)
            names[n] = kKernelNames[i];
        if (ms)
            ms[n] = h->prof_ms[i];
        if (launches)
            launches[n] = h->prof_n[i];
        n++;
    }
    if (reset) {
        memset(h->prof_ms, 0, sizeof(h->prof_ms));
        memset(h->prof_n, 0, sizeof(h->prof_n));
        cudaMemset(h->d_counters, 0, sizeof(unsigned long long) * (8 + 512));
    }
    return n;
}

long long cedar_b200_launch_count(cedar_b200_handle *h) { return h ? h->launches : 0; }

void *cedar_b200_stream(cedar_b200_handle *h) { return h ? (void *)h->stream : nullptr; }

long long cedar_b200_debug_read(cedar_b200_handle *h, int what, void *dst, size_t cap)
{
    if (!h || !dst || h->pipe)
        return -EINVAL;
    cudaSetDevice(h->device);
    const Geom &g = h->g;
    const void *src = nullptr;
    size_t n = 0;
    switch (what) {
    case 0: src = h->d_src[h->last_par], n = g.frame_bytes; break;
    case 1: src = h->d_unf, n = g.frame_bytes; break;
    case 2: src = h->d_rec[h->last_cur], n = g.frame_bytes; break;
    case 3: src = h->d_mbi[h->last_par], n = sizeof(MbInfo) * g.nmb; break;
    case 4: src = h->d_nnz[h->last_par], n = (size_t)NNZ_STRIDE * g.nmb; break;
    case 5: src = h->d_coef[h->last_par], n = sizeof(int16_t) * COEF_STRIDE * g.nmb; break;
    case 7: src = h->d_i4[h->last_par], n = (size_t)16 * g.nmb; break;
    case 6: src = h->eb.bins_len, n = sizeof(uint32_t) * (h->last_nframes > 0 ? h->last_nframes : 1) * h->S; break;
    case 8: src = h->d_counters, n = sizeof(unsigned long long) * (8 + 512); break;
    default: return -EINVAL;
    }
    if (n > cap)
        return -ENOMEM;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(dst, src, n, cudaMemcpyDeviceToHost));
    return (long long)n;
}

void cedar_b200_close(cedar_b200_handle *h)
{
    if (!h)
        return;
    cudaSetDevice(h->device);
    if (!h->pipe)
        prof_collect(h);
    double total_ns = std::chrono::duration<double, std::nano>(std::chrono::steady_clock::now() - h->t_open).count();
    // cedar.c:715-719 prints "Time spent: <waiting>/<total>ns" at release
    fprintf(stderr, "cedar_b200: Time spent: %.0f/%.0fns\n", h->busy_ns, total_ns);
    destroy_handle(h);
}

} // extern "C"
