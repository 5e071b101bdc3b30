// sm_100a CUDA kernels of the B200 H.264 encoder: the replacement for the Cedar VE frame encode that
// the reference triggers with one register write (kernel/cedar.c:1176) and has no source for.
// Row numbers K0..K9 are SURVEY.md 8a's kernel rows.  None of this is a dense contraction, so
// there are no tensor-core instructions here: integer SIMD-video (VABSDIFF4) for motion search,
// HBM / L2 streaming and dependency-ordered wavefronts for everything else.
//
// Many closed GOPs ("lanes") are encoded in lock step: blockIdx.y = lane (me_kernel: blockIdx.z), lane l holds stream
// frame step.frame0 + l * step.lane_stride.
#pragma once
#include "entropy.cuh"
#include <cstdio>

namespace cedar {

struct Step {
    int nlanes;      // lanes launched
    int frame0;      // clip frame index held by lane 0
    int lane_stride; // frames between consecutive lanes (the GOP length)
    int nframes;     // frames in the clip; lanes beyond it idle
};
__device__ __forceinline__ int lane_frame(const Step &s, int lane)
{
    int f = s.frame0 + lane * s.lane_stride;
    return f < s.nframes ? f : -1;
}

// Wavefront progress flags: the producer warp stores its pixels, __syncwarp()s, and lane 0 publishes
// the count with a gpu-scope release; the consumer's lane 0 spins with acquire loads, __syncwarp()s, and
// the warp then reads the neighbour's pixels from L2 (__ldcg).
__device__ __forceinline__ int ld_acquire(const int *p)
{
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int *p, int v)
{
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// ================================================================================================
// K0 ingest: packed NV12 / NV16 (w x h) -> planar 4:2:0 at the coded size with edge replication.
// Replaces the ISP input stage (cedar.c:1068-1080).  Grid: (16-byte groups of a luma row / 128, H + 2 CH output rows,
// lanes); one thread = 16 output bytes: one aligned 16-byte vector of luma, or two vectors of interleaved chroma
// de-interleaved with byte permutes (NV16: the rounding average of two rows, __vavgu4); words and bytes only at the
// picture edge or when the source is not 16-byte aligned.  HBM bound.
// ================================================================================================
__device__ __forceinline__ uint32_t ingest_luma_word(const uint8_t *rp, int x, int src_w)
{
    if (x + 3 < src_w && !((uintptr_t)(rp + x) & 3))
        return *(const uint32_t *)(rp + x);
    uint32_t out = 0;
#pragma unroll
    for (int k = 0; k < 4; k++)
        out |= (uint32_t)rp[imin_(x + k, src_w - 1)] << (8 * k);
    return out;
}
__device__ __forceinline__ uint32_t ingest_chroma_word(const uint8_t *ra, const uint8_t *rb, int x, int c, int src_w, int nv16)
{
    uint32_t out = 0;
    if (2 * x + 7 < src_w && !(((uintptr_t)(ra + 2 * x) | (uintptr_t)(rb + 2 * x)) & 3)) {
        const uint32_t sel = c ? 0x7531u : 0x6420u;
        const uint32_t *pa = (const uint32_t *)(ra + 2 * x), *pb = (const uint32_t *)(rb + 2 * x);
        out = __byte_perm(pa[0], pa[1], sel);
        if (nv16)
            out = __vavgu4(out, __byte_perm(pb[0], pb[1], sel));
    } else {
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int sx = imin_(x + k, src_w / 2 - 1);
            const int a = ra[2 * sx + c], b = rb[2 * sx + c];
            out |= (uint32_t)((a + b + 1) >> 1) << (8 * k);
        }
    }
    return out;
}
__global__ void __launch_bounds__(128) ingest_kernel(Geom g, Step s, const uint8_t *__restrict__ raw, size_t raw_frame_bytes,
                                                     uint8_t *__restrict__ src)
{
    const int f = lane_frame(s, blockIdx.z);
    if (f < 0)
        return;
    const int row = blockIdx.y, x = (blockIdx.x * 128 + threadIdx.x) * 16;
    const uint8_t *luma = raw + (size_t)f * raw_frame_bytes;
    const uint8_t *chroma = luma + (size_t)g.src_w * g.src_h;
    uint8_t *dst = src + (size_t)blockIdx.z * g.frame_bytes;
    uint4 out;
    if (row < g.H) {
        if (x >= g.W)
            return;
        const uint8_t *rp = luma + (size_t)imin_(row, g.src_h - 1) * g.src_w;
        if (x + 15 < g.src_w && !((uintptr_t)(rp + x) & 15))
            out = *(const uint4 *)(rp + x);
        else
            out = make_uint4(ingest_luma_word(rp, x, g.src_w), ingest_luma_word(rp, x + 4, g.src_w),
                             ingest_luma_word(rp, x + 8, g.src_w), ingest_luma_word(rp, x + 12, g.src_w));
        *(uint4 *)(dst + (size_t)row * g.W + x) = out; // W is a multiple of 16
    } else {
        if (x >= g.CW)
            return;
        const int cr = row - g.H, c = cr >= g.CH, y = cr - (c ? g.CH : 0);
        const int sy = imin_(y, g.src_h / 2 - 1), nv16 = g.src_format == 1;
        // NV16 -> 4:2:0: rounding average of the two chroma rows
        const uint8_t *ra = chroma + (size_t)(nv16 ? 2 * sy : sy) * g.src_w, *rb = nv16 ? ra + g.src_w : ra;
        uint8_t *o = dst + (size_t)g.W * g.H + (size_t)c * g.CW * g.CH + (size_t)y * g.CW + x;
        if (x + 15 < g.CW && 2 * x + 31 < g.src_w && !(((uintptr_t)(ra + 2 * x) | (uintptr_t)(rb + 2 * x) | (uintptr_t)o) & 15)) {
            const uint32_t sel = c ? 0x7531u : 0x6420u;
            const uint4 a0 = ((const uint4 *)(ra + 2 * x))[0], a1 = ((const uint4 *)(ra + 2 * x))[1];
            out = make_uint4(__byte_perm(a0.x, a0.y, sel), __byte_perm(a0.z, a0.w, sel), __byte_perm(a1.x, a1.y, sel),
                             __byte_perm(a1.z, a1.w, sel));
            if (nv16) {
                const uint4 b0 = ((const uint4 *)(rb + 2 * x))[0], b1 = ((const uint4 *)(rb + 2 * x))[1];
                out.x = __vavgu4(out.x, __byte_perm(b0.x, b0.y, sel));
                out.y = __vavgu4(out.y, __byte_perm(b0.z, b0.w, sel));
                out.z = __vavgu4(out.z, __byte_perm(b1.x, b1.y, sel));
                out.w = __vavgu4(out.w, __byte_perm(b1.z, b1.w, sel));
            }
            *(uint4 *)o = out; // (CW is a multiple of 8 only: rows of some sizes start 8-byte aligned and take the word path)
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (x + 4 * k < g.CW)
                    *(uint32_t *)(o + 4 * k) = ingest_chroma_word(ra, rb, x + 4 * k, c, g.src_w, nv16);
        }
    }
}

// ================================================================================================
// K1 integer motion estimation: exhaustive +-R SAD search against the previous deblocked
// reconstruction (edge clamped).  One CTA per tile of nstrip x me_rows macroblocks (4 x 4 at R <= 32) that share
// one search window.  The window is staged in shared memory four times, byte-shifted by 0..3, so that every
// candidate reads aligned 32-bit words; a warp task = 32 column offsets x 4 consecutive row offsets of one
// macroblock: each thread streams that macroblock's 16x16 block through registers and issues 256
// VABSDIFF4-with-accumulate for 76 window loads.  argmin over key = cost << 15 | raster rank
// (order independent => deterministic).  Bound: integer SIMD-video issue rate.
// ================================================================================================
#define ME_THREADS 320
#define ME_MAX_STRIP 4
#define ME_MAX_ROWS 4 // macroblock rows per CTA (me_rows): they share 2R of the 16 + 2R window rows each would stage alone
#define ME_MAX_MB (ME_MAX_STRIP * ME_MAX_ROWS)
#define ME_TASK_WORDS 1088 // 32-column x 4-row tasks of one tile: at most 16 macroblocks x 2 x 17 (R = 32); R = 64: 2 x 4 x 33

__device__ __forceinline__ uint32_t sad4_acc(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("vabsdiff4.u32.u32.u32.add %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

__host__ __device__ inline int me_strip(int R) { return R > 32 ? 2 : ME_MAX_STRIP; }
__host__ __device__ inline int me_rows(int R) { return R > 32 ? 1 : ME_MAX_ROWS; } // shared memory: 4 CTAs per SM at R = 16, 2 at R = 64
__host__ __device__ inline int me_row_words(int R, int nstrip)
{
    int w = (16 * nstrip + 2 * R + 3) / 4 + 2;
    return w | 1; // odd: consecutive row groups of the transposed (left-over column) tasks hit different banks
}
__host__ __device__ inline int me_window_rows(int R) { return 16 * me_rows(R) + 2 * R + (R < 2 ? 3 : 0); } // R = 1: see me_group_row
__host__ __device__ inline int me_copy_words(int R, int nstrip)
{
    int cw = me_window_rows(R) * me_row_words(R, nstrip);
    return cw + ((8 - (cw & 31)) & 31); // == 8 (mod 32): the four copies start 8 banks apart
}
__host__ __device__ inline int me_item_words(int R, int nstrip) // left-over column items, padded to whole warps
{
    int nd = 2 * R + 1;
    return (((nd & 31) * ((nd + 3) >> 2) * nstrip * me_rows(R)) + 31) & ~31;
}
// Host side of me_kernel's tables: [0, 136) lambda * bits(offset - R),
// [136, 136 + 528) task table entries macroblock | column offset << 4 | first row offset << 12, then the left-over items.
// Macroblock m of a CTA = column m % nstrip, row m / nstrip of its nstrip x me_rows(R) tile.
// A task covers four consecutive row offsets; the last group of a column is moved up to end at the last offset (it
// repeats up to three candidates of the group before it, which cannot change an argmin), so no candidate lies outside
// the range -- except the fourth one when there are only three offsets (R = 1), which the kernel discards.
inline int me_group_row(int group, int nd) // first row offset of a group of four
{
    int oy0 = 4 * group;
    return oy0 + 4 <= nd ? oy0 : (nd >= 4 ? nd - 4 : 0);
}
inline size_t me_table_words(int R, int nstrip) { return 136 + ME_TASK_WORDS + me_item_words(R, nstrip); }
inline void me_build_tables(int R, int nstrip, int lambda, uint32_t *t)
{
    const int nd = 2 * R + 1, nfull = nd >> 5, nleft = nd & 31, ndyg = (nd + 3) >> 2, ntask_full = nfull * ndyg;
    for (int i = 0; i < 136; i++) {
        int d = i - R, a = d < 0 ? -d : d, bits = 1;
        if (a) {
            int lg = 0;
            while ((a >> lg) > 1)
                lg++;
            bits = 7 + 2 * lg;
        }
        t[i] = (uint32_t)(lambda * bits);
    }
    uint32_t *task = t + 136, *item = task + ME_TASK_WORDS;
    const int nmb = nstrip * me_rows(R);
    for (int i = 0; i < ntask_full * nmb; i++) {
        int m = i / ntask_full, k = i - m * ntask_full;
        task[i] = (uint32_t)m | ((uint32_t)((k / ndyg) * 32) << 4) | ((uint32_t)me_group_row(k % ndyg, nd) << 12);
    }
    const int per_mb = nleft * ndyg;
    for (int i = 0; i < me_item_words(R, nstrip); i++) {
        int m = per_mb ? i / per_mb : 0, jj = i - m * per_mb;
        item[i] = (per_mb && m < nmb) ? (uint32_t)m | ((uint32_t)(nfull * 32 + jj / ndyg) << 4) |
                                               ((uint32_t)me_group_row(jj % ndyg, nd) << 12)
                                         : 0xffffffffu;
    }
}
__host__ __device__ inline size_t me_smem_bytes(int R, int nstrip)
{
    return (size_t)(64 * nstrip * me_rows(R) + 4 * me_copy_words(R, nstrip) + me_item_words(R, nstrip)) * 4;
}

// Block-sum bound of the search (R <= 32, 4 x 4 tiles).  Split each 16 x 16 block into its sixteen 4 x 4 sub-blocks with
// pixel sums A_g (current) and B_g (candidate).  |A - B| >= 16 |floor(A / 16) - floor(B / 16)| - 15, so
//     SAD >= 16 * sum_g |floor(A_g / 16) - floor(B_g / 16)| - 240,
// and the quantised sums are bytes: four VABSDIFF4 bound a candidate whose SAD takes 64.  The quantised sums of every
// 4 x 4 window position are one table per CTA, built from the staged window; the table and the list of candidates whose
// bound does not rule them out live in the space of the three byte-shifted window copies, which the bound path does not
// stage (it reads copy 0 with funnel shifts).  Table row y holds four phase rows (x mod 4) of tpw words; byte b of phase
// row c is the position x = 4 b + c, so one unaligned word of it is the four sub-block columns of a candidate.
#define ME_LIST_CAP 2048 // candidates per tile that the SAD stage takes; a tile with more runs the exhaustive search
__host__ __device__ inline int me_tab_pw(int R, int nstrip) { return ((16 * (nstrip - 1) + 2 * R + 12) >> 4) + 2; }
__host__ __device__ inline int me_tab_rows(int R) { return me_window_rows(R) - 3; }
// three more rows (zero) for the row offsets past the range that the bound stage's lanes run through
__host__ __device__ inline int me_tab_words(int R, int nstrip) { return (me_tab_rows(R) + 3) * 4 * me_tab_pw(R, nstrip); }
inline bool me_bound_path(int R) // the geometries that take the bound path; the rest search exhaustively
{
    if (R < 2 || R > 32) // R < 2: fewer than four row offsets; R > 32: 2 x 1 tiles, whose window leaves no room
        return false;
    const int nstrip = me_strip(R);
    return 4 * nstrip * me_rows(R) + me_tab_words(R, nstrip) + ME_LIST_CAP <= 3 * me_copy_words(R, nstrip);
}

// Everything about the search geometry that only depends on the configuration, computed once on the host: the kernel's
// prologue runs once per warp and 200 k warps per launch make every division in it count.
struct MeShape {
    int nstrip, lstrip, nrow, RSW, CWs, WR, nd, nfull, nleft, ndyg; // lstrip = log2(nstrip)
    int bound;                       // block-sum bound path (me_bound_path)
    int tpw, trows;                  // its table: words per phase row, rows
    int tseg, tnseg;                 // its build: rows per segment, segments (one pass of the CTA's threads, me_shape)
    uint32_t nd_magic;               // __umulhi(i, nd_magic) == i / nd for the bound stage's item indices
    int noprune;                     // measurement only (CEDAR_B200_NO_PRUNE): every candidate is accumulated to the end
    // measurement only (profiling on), else null: [0] executed VABSDIFF4 lane-instructions, [1] candidates bounded,
    // [2] candidates that reached the SAD stage, [3] tiles on the bound path, [4] of them, tiles that searched exhaustively
    unsigned long long *exec_count;
};
inline MeShape me_shape(int R)
{
    MeShape m;
    m.nstrip = me_strip(R);
    m.lstrip = m.nstrip == 4 ? 2 : 1;
    m.nrow = me_rows(R);
    m.RSW = me_row_words(R, m.nstrip);
    m.CWs = me_copy_words(R, m.nstrip);
    m.WR = me_window_rows(R);
    m.nd = 2 * R + 1;
    m.nfull = m.nd >> 5, m.nleft = m.nd & 31, m.ndyg = (m.nd + 3) >> 2;
    m.bound = me_bound_path(R);
    m.tpw = me_tab_pw(R, m.nstrip);
    m.trows = me_tab_rows(R);
    // the table build's thread = (segment, phase, word): the shortest segments that still give every thread at most one
    // item (R = 16: 11 segments of 9 rows x 28 words = 308 items), so the CTA builds the table in one pass
    const int tw = 4 * m.tpw, per_col = ME_THREADS / tw > 0 ? ME_THREADS / tw : 1;
    m.tseg = (m.trows + per_col - 1) / per_col;
    m.tnseg = (m.trows + m.tseg - 1) / m.tseg;
    m.nd_magic = (uint32_t)(((1ull << 32) + (unsigned)m.nd - 1) / (unsigned)m.nd); // exact for i < 2^32 / nd
    m.noprune = 0;
    m.exec_count = nullptr;
    return m;
}

// Grid: (strips per macroblock row, macroblock rows / me_rows, lanes).
// kRSW: words per window row as a compile-time constant (the offsets of the unrolled search loop become immediates:
// 14 % fewer instructions), 0 = any geometry.
// kCount: the measurement build of the same kernel (profiling on): counts the executed VABSDIFF4 lane-instructions and
// honours MeShape::noprune; the product launches kCount = false, which carries neither.
template <int kRSW, bool kCount = false>
__global__ void __launch_bounds__(ME_THREADS, kCount ? 1 : 4) me_kernel(Geom g, Step s, MeShape ms, const uint8_t *__restrict__ src,
                                                       const uint8_t *__restrict__ ref, MbInfo *__restrict__ mbi,
                                                       const MbInfo *__restrict__ mbi_prev,
                                                       const uint32_t *__restrict__ tabs)
{
    extern __shared__ uint32_t sm[];
    __shared__ uint32_t mb_best[ME_MAX_MB];
    __shared__ uint32_t mvcost[136];      // lambda * bits(offset - R)
    __shared__ uint32_t task_tab[ME_TASK_WORDS];
    __shared__ int list_n; // bound path: candidates that passed the bound
    if (lane_frame(s, blockIdx.z) < 0)
        return;
    const int R = g.R, nd = ms.nd, nstrip = ms.nstrip;
    const int WR = ms.WR, RSW = kRSW ? kRSW : ms.RSW, CWs = ms.CWs;
    const int mby0 = blockIdx.y * ms.nrow, mbx0 = blockIdx.x * nstrip, nmb = nstrip * ms.nrow, ls = ms.lstrip;
    const int ncols = imin_(nstrip, g.mbw - mbx0), nrows = imin_(ms.nrow, g.mbh - mby0); // the tile may hang over the picture
    uint32_t vmask = 0; // macroblocks of the tile that exist
#pragma unroll
    for (int m = 0; m < ME_MAX_MB; m++)
        vmask |= (uint32_t)(m < nmb && (m & (nstrip - 1)) < ncols && (m >> ls) < nrows) << m;
    const int x0 = mbx0 * 16, y0 = mby0 * 16;
    const uint8_t *srcY = src + (size_t)blockIdx.z * g.frame_bytes;
    const uint8_t *refY = ref + (size_t)blockIdx.z * g.frame_bytes;
    uint32_t *cur_s = sm, *cp = sm + 64 * nmb, *item_tab = cp + 4 * CWs;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nwarps = ME_THREADS / 32;
#ifdef ME_PROFILE
    // Measurement build (-DME_PROFILE): clock64 marks at the phase boundaries, behind a barrier so that a phase ends when
    // its slowest warp does; thread 0 adds them to exec_count[480 + phase] and counts the tile in exec_count[487]
    unsigned long long prof_pt[7] = {0, 0, 0, 0, 0, 0, 0};
    long long prof_t = clock64();
#define ME_MARK(i)                                                                                                     \
    {                                                                                                                  \
        __syncthreads();                                                                                               \
        const long long now_ = clock64();                                                                              \
        prof_pt[i] += (unsigned long long)(now_ - prof_t);                                                             \
        prof_t = now_;                                                                                                 \
    }
#else
#define ME_MARK(i)
#endif

    // Tables that take every division and every bit-length computation out of the task loop; they only depend on the
    // configuration, so the host builds them once (me_build_tables) and every CTA copies them; tasks of macroblocks
    // beyond the picture edge are skipped (vmask).  The task tables are read by the exhaustive search only: a tile on
    // the bound path copies them when its list overflows.
    const int nleft = ms.nleft, ndyg = ms.ndyg;
    const int ntask_full = ms.nfull * ndyg;               // per macroblock: 32 columns x one row group
    const int nitems_left = nleft * ndyg * nmb;        // left-over columns of all macroblocks, one item per lane
    auto copy_task_tables = [&]() {
        for (int i = tid; i < ntask_full * nmb; i += ME_THREADS)
            task_tab[i] = tabs[136 + i];
        for (int i = tid; i < ((nitems_left + 31) & ~31); i += ME_THREADS)
            item_tab[i] = i < nitems_left ? tabs[136 + ME_TASK_WORDS + i] : 0xffffffffu;
    };
    const bool bound = kRSW != 43 && ms.bound; // kRSW = 43 is R > 32, never on the bound path

    // Window staging: warp = window row (round robin), lane = 32-bit word of the row.  Each lane fetches its
    // word and the next one (the second fetch hits L1) and builds the three byte-shifted copies in
    // registers; no integer division, no shared-memory round trip.  plain: copy 0, shifted: copies 1..3.
    // Interior tiles whose window starts on a 16-byte boundary (R = 16: all of them), is at most 32 words wide and at
    // most three passes tall: eight lanes per row, four rows per warp pass, one 16-byte load per lane -- a third of the
    // instructions of the word-per-lane loop.  The four rows of a pass land in different banks (RSW is odd).  The
    // loads of all passes are issued before the first store (vec_load), so a lane waits for one round trip, not three.
    const bool interior_x = x0 - R >= 0 && x0 - R + 4 * RSW + 4 <= g.W && !((x0 - R) & 3);
    const int nq = (RSW + 4) >> 2; // 16-byte groups that hold window words 0 .. RSW
    constexpr int kPasses = 3;
    const bool vec = interior_x && !((x0 - R) & 15) && RSW < 32 && x0 - R + 16 * nq <= g.W && WR <= 4 * nwarps * kPasses;
    auto vec_load = [&](uint4 *v) {
#pragma unroll
        for (int p = 0; p < kPasses; p++) {
            const int r = 4 * (warp + nwarps * p) + (lane >> 3), q = lane & 7;
            v[p] = make_uint4(0, 0, 0, 0);
            if (vec && r < WR && q < nq)
                v[p] = *(const uint4 *)(refY + (size_t)clip3_(0, g.H - 1, y0 - R + r) * g.W + (x0 - R) + 16 * q);
        }
    };
    auto stage = [&](const uint4 *v, const bool plain, const bool shifted) {
        auto fetch = [&](const uint8_t *row, int k) -> uint32_t { // window word k of a row, edge clamped
            const int fx = x0 - R + 4 * k;
            if (interior_x)
                return *(const uint32_t *)(row + fx);
            uint32_t v = 0;
#pragma unroll
            for (int i = 0; i < 4; i++)
                v |= (uint32_t)row[clip3_(0, g.W - 1, fx + i)] << (8 * i);
            return v;
        };
        if (vec) {
            const int sub = lane >> 3, q = lane & 7;
#pragma unroll
            for (int p = 0; p < kPasses; p++) {
                const int r = 4 * (warp + nwarps * p) + sub;
                const bool on = r < WR && q < nq;
                const uint32_t w[5] = {v[p].x, v[p].y, v[p].z, v[p].w, __shfl_down_sync(0xffffffffu, v[p].x, 1)};
                uint32_t *d = cp + r * RSW + 4 * q;
#pragma unroll
                for (int i = 0; i < 4; i++)
                    if (on && 4 * q + i < RSW) {
                        if (plain)
                            d[i] = w[i];
                        if (shifted) {
                            d[i + CWs] = __byte_perm(w[i], w[i + 1], 0x4321);
                            d[i + 2 * CWs] = __byte_perm(w[i], w[i + 1], 0x5432);
                            d[i + 3 * CWs] = __byte_perm(w[i], w[i + 1], 0x6543);
                        }
                    }
            }
        }
        for (int r = vec ? WR : warp; r < WR; r += ME_THREADS / 32) {
            const uint8_t *row = refY + (size_t)clip3_(0, g.H - 1, y0 - R + r) * g.W;
            for (int k0 = 0; k0 < RSW; k0 += 32) {
                const int k = k0 + lane;
                const uint32_t lo = k <= RSW ? fetch(row, k) : 0u;
                uint32_t hi = __shfl_down_sync(0xffffffffu, lo, 1); // the next word is the neighbouring lane's
                if (lane == 31 && k < RSW)
                    hi = fetch(row, k + 1);
                if (k < RSW) {
                    uint32_t *d = cp + r * RSW + k;
                    if (plain)
                        d[0] = lo;
                    if (shifted) {
                        d[CWs] = __byte_perm(lo, hi, 0x4321);
                        d[2 * CWs] = __byte_perm(lo, hi, 0x5432);
                        d[3 * CWs] = __byte_perm(lo, hi, 0x6543);
                    }
                }
            }
        }
    };
    // One round of global loads per thread, all issued before its first shared store: a word of the vector-cost table,
    // a 16-byte row of a current block ([mb][row][4 words]: thread = mb * 16 + row), the window rows of its warp and the
    // motion vectors of the seeds' co-located macroblocks (one warp pass per macroblock, at most two per warp).
    static_assert(ME_MAX_MB * 16 <= ME_THREADS && ME_MAX_MB <= 2 * (ME_THREADS / 32), "me_kernel: one load round");
    const uint32_t cost_w = tid < 136 ? tabs[tid] : 0u;
    uint4 cur_w = make_uint4(0, 0, 0, 0);
    const bool cur_on = tid < 16 * nmb && ((vmask >> (tid >> 4)) & 1);
    if (cur_on) {
        const int m = tid >> 4;
        cur_w = *(const uint4 *)(srcY + (size_t)(y0 + 16 * (m >> ls) + (tid & 15)) * g.W + x0 + 16 * (m & (nstrip - 1)));
    }
    uint4 wv[kPasses];
    vec_load(wv);
    int seed_mv[2] = {0, 0}; // mv[0] | mv[1] << 16 of MbInfo
#pragma unroll
    for (int k = 0; k < 2; k++) {
        const int m = warp + nwarps * k;
        if (lane >= 16 && m < nmb && ((vmask >> m) & 1))
            seed_mv[k] = *(const int *)mbi_prev[(size_t)blockIdx.z * g.nmb + (size_t)(mby0 + (m >> ls)) * g.mbw + mbx0 +
                                                 (m & (nstrip - 1))].mv;
    }
    if (tid < 136)
        mvcost[tid] = cost_w;
    if (cur_on)
        ((uint4 *)cur_s)[tid] = cur_w;
    if (tid < ME_MAX_MB)
        mb_best[tid] = 0xffffffffu;
    if (tid == 0)
        list_n = 0;
    if (!bound)
        copy_task_tables();
    ME_MARK(0);
    stage(wv, true, !bound);
    __syncthreads();
    ME_MARK(1);
    // copy 0 read at byte offset ox & 3 (what copy ox & 3 holds): the seeds and the bound path's SAD stage
    auto win = [&](const uint32_t *p, int sh) { return __funnelshift_r(p[0], p[1], sh); };
    unsigned nabs = 0; // measurement build: VABSDIFF4 lane-instructions of the bound path

    // Seed the running minimum with two real candidates per macroblock -- the zero vector and the vector the
    // co-located macroblock had in the previous frame (any value is fine: it only has to be a candidate of the
    // search) -- so that the bound stage can reject candidates outright and the SAD loops can drop a task as soon as the
    // partial cost of every candidate in it exceeds the best complete cost so far.  SAD terms are non-negative, so the partial key is a lower
    // bound of the final key: the argmin, and with it the bitstream, is unchanged.
    // one warp pass per macroblock: lanes 0..15 take the rows of the zero-vector seed, lanes 16..31 those of the
    // co-located one
#pragma unroll
    for (int k = 0; k < 2; k++) {
        const int m = warp + nwarps * k;
        const int mc = m & (nstrip - 1), mr = m >> ls, half = lane >> 4, l16 = lane & 15;
        if (m >= nmb || !((vmask >> m) & 1))
            continue;
        int ox = R, oy = R;
        if (half) {
            ox = clip3_(0, nd - 1, ((int)(int16_t)seed_mv[k] >> 2) + R);
            oy = clip3_(0, nd - 1, (seed_mv[k] >> 18) + R);
        }
        uint32_t a = 0;
        const uint32_t *wp = cp + (oy + 16 * mr + l16) * RSW + 4 * mc + (ox >> 2);
        const uint32_t *cu = cur_s + 64 * m + 4 * l16;
#pragma unroll
        for (int k = 0; k < 4; k++)
            a = sad4_acc(win(wp + k, 8 * (ox & 3)), cu[k], a);
        a = __reduce_add_sync(half ? 0xffff0000u : 0x0000ffffu, a);
        if (l16 == 0)
            atomicMin(&mb_best[m], ((a + mvcost[ox] + mvcost[oy]) << 15) | (uint32_t)(oy * nd + ox));
    }
    // Bound path: the quantised 4 x 4 sums of the current blocks (word 4 m + i = sub-block row i of macroblock m, byte j =
    // sub-block column j) and of every window position (tab, see me_tab_pw)
    uint32_t *const qcur = cp + CWs, *const tab = qcur + 4 * nmb, *const list = tab + (ms.trows + 3) * 4 * ms.tpw;
    const int tpw = ms.tpw, tw = 4 * tpw;
    if (bound) {
        if (tid < 4 * nmb && ((vmask >> (tid >> 2)) & 1)) {
            const uint32_t *cu = cur_s + 16 * tid;
            uint32_t q = 0;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                uint32_t a = 0;
#pragma unroll
                for (int r = 0; r < 4; r++)
                    a = sad4_acc(cu[4 * r + j], 0u, a);
                q |= (a >> 4) << (8 * j);
            }
            qcur[tid] = q;
            if (kCount)
                nabs += 16;
        }
        for (int i = tid; i < 3 * tw; i += ME_THREADS)
            tab[ms.trows * tw + i] = 0;
        // thread = (segment of ms.tseg table rows, phase c, word w): four running rows of 4-pixel sums per column, so
        // every window word is read once per segment.  Bytes of positions no candidate reaches are 0.
        const int xs_max = 16 * (nstrip - 1) + 2 * R + 12;
        for (int it = tid; it < ms.tnseg * tw; it += ME_THREADS) {
            const int seg = it / tw, col = it - seg * tw, c = col / tpw, w = col - c * tpw;
            const int y0 = seg * ms.tseg, y1 = imin_(y0 + ms.tseg, ms.trows), sh = 8 * c;
            int idx[4];
            uint32_t valid = 0;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                idx[j] = imin_(4 * w + j, RSW - 2);
                valid |= (16 * w + c + 4 * j <= xs_max ? 0xffu : 0u) << (8 * j);
            }
            auto hrow = [&](int y, uint32_t *hh) {
#pragma unroll
                for (int j = 0; j < 4; j++)
                    hh[j] = sad4_acc(win(cp + y * RSW + idx[j], sh), 0u, 0u);
            };
            auto put = [&](int y, const uint32_t *a, const uint32_t *b, const uint32_t *c_, const uint32_t *d) {
                uint32_t q = 0;
#pragma unroll
                for (int j = 0; j < 4; j++)
                    q |= ((a[j] + b[j] + c_[j] + d[j]) >> 4) << (8 * j);
                tab[y * tw + col] = q & valid;
            };
            uint32_t h0[4], h1[4], h2[4], h3[4];
            hrow(y0, h0), hrow(y0 + 1, h1), hrow(y0 + 2, h2);
            for (int y = y0; y < y1; y += 4) {
                hrow(y + 3, h3), put(y, h0, h1, h2, h3);
                if (y + 1 < y1)
                    hrow(y + 4, h0), put(y + 1, h1, h2, h3, h0);
                if (y + 2 < y1)
                    hrow(y + 5, h1), put(y + 2, h2, h3, h0, h1);
                if (y + 3 < y1)
                    hrow(y + 6, h2), put(y + 3, h3, h0, h1, h2);
            }
            if (kCount)
                nabs += 4 * (y1 - y0 + 3);
        }
    }
    __syncthreads();
    ME_MARK(2);
    bool fallback = !bound;
    unsigned nbounded = 0, nsad = 0; // measurement build
    if (bound) {
        // Bound stage: item = (macroblock m, row phase c, column offset ox); a lane walks the row offsets c, c + 4, ..
        // and keeps the three table rows the next candidate shares.  A candidate whose bound key exceeds the best key
        // of the seeds cannot be the argmin (its key is at least the bound key); the others go to the list.
        const int nitem = nmb * 4 * nd;
        for (int i0 = warp * 32; i0 < nitem; i0 += nwarps * 32) {
            if (__shfl_sync(0xffffffffu, *(volatile int *)&list_n, 0) > ME_LIST_CAP)
                break; // the tile searches exhaustively: no need to bound the rest
            const int i = i0 + lane, t = (int)__umulhi((uint32_t)i, ms.nd_magic), ox = i - t * nd, c = t & 3;
            const bool live = i < nitem && ((vmask >> (t >> 2)) & 1);
            const int m = live ? t >> 2 : 0, x = 16 * (m & (nstrip - 1)) + ox, sh = 8 * ((x >> 2) & 3);
            // no branch per candidate: every lane runs ndyg row offsets (the table has rows for the ones past the range,
            // whose results are masked off) and sets bit j of pm when row offset c + 4 j passes
            const uint32_t *tp = tab + (16 * (m >> ls) + c) * tw + (x & 3) * tpw + (x >> 4);
            const uint4 q = ((const uint4 *)qcur)[m];
            const uint32_t best = mb_best[m], cx = mvcost[ox] - 240u; // cost = max(16 sb, 240) - 240 + mv cost
            uint32_t w0 = win(tp, sh), w1 = win(tp + 4 * tw, sh), w2 = win(tp + 8 * tw, sh), pm = 0;
            uint32_t rank = (uint32_t)(c * nd + ox);
            for (int j = 0; j < ndyg; j++) {
                const uint32_t w3 = win(tp + (4 * j + 12) * tw, sh);
                uint32_t sb = sad4_acc(w0, q.x, 0u);
                sb = sad4_acc(w1, q.y, sb);
                sb = sad4_acc(w2, q.z, sb);
                sb = sad4_acc(w3, q.w, sb);
                const uint32_t key = (max(16u * sb, 240u) + cx + mvcost[c + 4 * j]) * 32768u + rank;
                pm |= (uint32_t)(key <= best) << j;
                rank += 4u * (uint32_t)nd;
                w0 = w1, w1 = w2, w2 = w3;
            }
            pm &= live ? (1u << ((nd - c + 3) >> 2)) - 1u : 0u; // row offsets c + 4 j < nd
            if (kCount && live)
                nbounded += (nd - c + 3) >> 2;
            // append the passing candidates: one ballot and one shared atomic per round, a round per set bit
            while (__any_sync(0xffffffffu, pm)) {
                const bool pass = pm != 0;
                const int oy = c + 4 * (__ffs(pm) - 1);
                pm &= pm - 1;
                const uint32_t ball = __ballot_sync(0xffffffffu, pass);
                int base = 0;
                if (lane == 0)
                    base = atomicAdd(&list_n, __popc(ball));
                base = __shfl_sync(0xffffffffu, base, 0) + __popc(ball & ((1u << lane) - 1));
                if (pass && base < ME_LIST_CAP)
                    list[base] = (uint32_t)m | ((uint32_t)ox << 4) | ((uint32_t)oy << 12);
            }
        }
        if (kCount)
            nabs += 4 * nbounded;
        __syncthreads();
        ME_MARK(3);
        fallback = list_n > ME_LIST_CAP;
        if (!fallback) {
            // SAD stage: four lanes per listed candidate, eight candidates per warp pass, read from copy 0; lane l of a
            // candidate takes block rows l, l + 4, l + 8, l + 12 (four window words each by funnel shift, a chain of 16
            // VABSDIFF4), two shuffles sum them.  The key (cost << 15 | rank) does not depend on the order in which
            // candidates reach the minimum.
            const int n = list_n, sub = lane & 3;
            for (int i0 = 8 * warp; i0 < n; i0 += 8 * nwarps) {
                const int i = i0 + (lane >> 2);
                const uint32_t e = list[i < n ? i : i0]; // lanes past the list repeat the pass's first candidate
                const int m = (int)(e & 15), ox = (int)((e >> 4) & 255), oy = (int)(e >> 12), sh = 8 * (ox & 3);
                const uint32_t *wp = cp + (oy + 16 * (m >> ls) + sub) * RSW + 4 * (m & (nstrip - 1)) + (ox >> 2);
                const uint4 *cu = (const uint4 *)(cur_s + 64 * m) + sub;
                uint32_t a = 0;
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    const uint4 cw = cu[4 * r];
                    const uint32_t *p = wp + 4 * r * RSW;
                    a = sad4_acc(win(p, sh), cw.x, a);
                    a = sad4_acc(win(p + 1, sh), cw.y, a);
                    a = sad4_acc(win(p + 2, sh), cw.z, a);
                    a = sad4_acc(win(p + 3, sh), cw.w, a);
                }
                a += __shfl_xor_sync(0xffffffffu, a, 1);
                a += __shfl_xor_sync(0xffffffffu, a, 2);
                if (sub == 0 && i < n) {
                    atomicMin(&mb_best[m], ((a + mvcost[ox] + mvcost[oy]) << 15) | (uint32_t)(oy * nd + ox));
                    if (kCount)
                        nabs += 64, nsad++;
                }
            }
            ME_MARK(4);
        } else {
            // the exhaustive search below reads the task tables and the byte-shifted copies
            vec_load(wv);
            copy_task_tables();
            stage(wv, false, true);
            __syncthreads();
        }
    }
    if (kCount && ms.exec_count && bound) {
        const unsigned a = __reduce_add_sync(0xffffffffu, nabs), b = __reduce_add_sync(0xffffffffu, nbounded),
                       c = __reduce_add_sync(0xffffffffu, nsad);
        if (lane == 0) {
            atomicAdd(ms.exec_count, (unsigned long long)a);
            atomicAdd(ms.exec_count + 1, (unsigned long long)b);
            atomicAdd(ms.exec_count + 2, (unsigned long long)c);
        }
        if (tid == 0) {
            atomicAdd(ms.exec_count + 3, 1ull);
            atomicAdd(ms.exec_count + 4, (unsigned long long)fallback);
        }
    }
    // Exhaustive search: every geometry off the bound path, and bound-path tiles whose list overflowed
    const int ntask = fallback ? ntask_full * nmb + ((nitems_left + 31) >> 5) : 0;
    for (int task = warp; task < ntask; task += nwarps) {
        // task table entry: macroblock | column offset << 4 | first row offset << 12 (0xffffffff = idle lane)
        const uint32_t e = task < ntask_full * nmb ? task_tab[task] + ((uint32_t)lane << 4)
                                                   : item_tab[(task - ntask_full * nmb) * 32 + lane];
        uint32_t key = 0xffffffffu;
        const int m = (int)(e & 15);
        if (e != 0xffffffffu && ((vmask >> m) & 1)) {
            const int ox = (int)((e >> 4) & 255), oy0 = (int)(e >> 12);
            uint32_t cur[64];
            {
                const uint4 *c4 = (const uint4 *)(cur_s + 64 * m);
#pragma unroll
                for (int i = 0; i < 16; i++) {
                    uint4 v = c4[i];
                    cur[4 * i] = v.x, cur[4 * i + 1] = v.y, cur[4 * i + 2] = v.z, cur[4 * i + 3] = v.w;
                }
            }
            const uint32_t *wp = cp + (ox & 3) * CWs + (oy0 + 16 * (m >> ls)) * RSW + 4 * (m & (nstrip - 1)) + (ox >> 2);
            // cost = SAD + lambda * (bits(mvx) + bits(mvy)): the accumulators start at the vector cost, so a key is one
            // multiply-add (cost << 15 | raster rank; cost < 2^17)
            const uint32_t cx = mvcost[ox], rank0 = (uint32_t)(oy0 * nd + ox);
            uint32_t acc[4] = {cx + mvcost[oy0], cx + mvcost[oy0 + 1], cx + mvcost[oy0 + 2], cx + mvcost[oy0 + 3]};
            auto min_key = [&]() {
                uint32_t pm = 0xffffffffu;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    uint32_t k = acc[j] * 32768u + (rank0 + (uint32_t)(j * nd));
                    if (j == 3 && nd < 4) // R = 1: there is no fourth row offset
                        k = 0xffffffffu;
                    pm = k < pm ? k : pm;
                }
                return pm;
            };
            bool dead = false;
            int rows_done = 19;
#pragma unroll
            for (int r = 0; r < 19; r++) {
                // partial keys (rows 0 .. r - 1 - j of candidate j) against the best complete key.  Measured on the
                // benchmark clip: 0.1 % of the tasks are dead after 5 window rows, 5 % after 9, 30 % after 13.
                // With a wide range (R = 64, kRSW = 43) most candidates are far from the match and the early check pays;
                // compile-time, because the extra branch point costs the R = 16 loop 20 % even when it is never taken.
                if ((r == 5 && kRSW == 43) || r == 9 || r == 13)
                    dead = min_key() > *(volatile uint32_t *)&mb_best[m] && !(kCount && ms.noprune);
                if (dead) {
                    if (kCount)
                        rows_done = r;
                    break;
                }
                uint32_t w0 = wp[r * RSW], w1 = wp[r * RSW + 1], w2 = wp[r * RSW + 2], w3 = wp[r * RSW + 3];
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    int cr = r - j; // candidate row offset oy0 + j compares window row r with block row r - j
                    if (cr >= 0 && cr < 16) {
                        acc[j] = sad4_acc(w0, cur[cr * 4 + 0], acc[j]);
                        acc[j] = sad4_acc(w1, cur[cr * 4 + 1], acc[j]);
                        acc[j] = sad4_acc(w2, cur[cr * 4 + 2], acc[j]);
                        acc[j] = sad4_acc(w3, cur[cr * 4 + 3], acc[j]);
                    }
                }
            }
            if (!dead)
                key = min_key();
            if (kCount && ms.exec_count) { // window rows 0 .. rows_done - 1: row r feeds min(r + 1, 4, 19 - r) candidates, four words each
                unsigned n4 = 0;
                for (int r = 0; r < rows_done; r++)
                    n4 += 4u * (unsigned)imin_(imin_(r + 1, 4), 19 - r);
                n4 = __reduce_add_sync(__activemask(), n4);
                if ((__activemask() & ((1u << lane) - 1)) == 0)
                    atomicAdd(ms.exec_count, (unsigned long long)n4);
            }
        }
        // the lanes of a full task share the macroblock; the left-over task mixes macroblocks
        if (task < ntask_full * nmb) {
            key = __reduce_min_sync(0xffffffffu, key);
            if (lane == 0)
                atomicMin(&mb_best[m], key);
        } else if (key != 0xffffffffu)
            atomicMin(&mb_best[m], key);
    }
    __syncthreads();
    ME_MARK(5);
    if (tid < nmb && ((vmask >> tid) & 1)) {
        const uint32_t b = mb_best[tid];
        int rank = (int)(b & 0x7fff);
        MbInfo mi;
        mi.type = MB_P16x16;
        mi.i16_mode = mi.chroma_mode = mi.cbp = 0;
        mi.mv[0] = (int16_t)((rank % nd - R) * 4);
        mi.mv[1] = (int16_t)((rank / nd - R) * 4);
        mi.mvd[0] = mi.mvd[1] = 0;
        mi.pad = b >> 15; // best cost, for statistics
        mbi[(size_t)blockIdx.z * g.nmb + (size_t)(mby0 + (tid >> ls)) * g.mbw + mbx0 + (tid & (nstrip - 1))] = mi;
    }
#ifdef ME_PROFILE
    ME_MARK(6);
    if (tid == 0 && ms.exec_count) {
        for (int i = 0; i < 7; i++)
            atomicAdd(ms.exec_count + 480 + i, prof_pt[i]);
        atomicAdd(ms.exec_count + 487, 1ull);
    }
#endif
#undef ME_MARK
}

// ================================================================================================
// Shared per-lane chroma path (used by the inter and intra kernels): lanes 16..23 of the warp
// own the eight 4x4 chroma blocks (16..19 Cb, 20..23 Cr).  `w` = forward-transformed residual.
// ================================================================================================
struct ChromaOut {
    int zdc;   // quantised DC level owned by this lane (index cb of its plane)
    int dcq;   // dequantised DC for this lane's block
    int cbpc;  // chroma CBP of the macroblock (warp uniform)
    unsigned m_dc; // ballot of non-zero DC levels
};

__device__ __forceinline__ ChromaOut chroma_dc_path(const int *w, int nz_ac, bool chroma, int lane, int qpc, int intra)
{
    ChromaOut o;
    const int base = 16 + ((lane - 16) & 4), cb = lane & 3;
    int d0 = __shfl_sync(0xffffffffu, w[0], base + 0), d1 = __shfl_sync(0xffffffffu, w[0], base + 1);
    int d2 = __shfl_sync(0xffffffffu, w[0], base + 2), d3 = __shfl_sync(0xffffffffu, w[0], base + 3);
    int qbits = 15 + qpc / 6, f = (1 << qbits) / (intra ? 3 : 6);
    o.zdc = chroma ? quant1(hadamard2x2_elem(cb, d0, d1, d2, d3), h264_quant_mf[qpc % 6][0], 2 * f, qbits + 1) : 0;
    unsigned m_ac = __ballot_sync(0xffffffffu, chroma && nz_ac > 0);
    o.m_dc = __ballot_sync(0xffffffffu, chroma && o.zdc != 0);
    o.cbpc = m_ac ? 2 : (o.m_dc ? 1 : 0);
    int z0 = __shfl_sync(0xffffffffu, o.zdc, base + 0), z1 = __shfl_sync(0xffffffffu, o.zdc, base + 1);
    int z2 = __shfl_sync(0xffffffffu, o.zdc, base + 2), z3 = __shfl_sync(0xffffffffu, o.zdc, base + 3);
    o.dcq = dequant_chroma_dc(hadamard2x2_elem(cb, z0, z1, z2, z3), qpc);
    return o;
}

__device__ __forceinline__ uint32_t pack4(const int *v)
{
    return (uint32_t)v[0] | ((uint32_t)v[1] << 8) | ((uint32_t)v[2] << 16) | ((uint32_t)v[3] << 24);
}

__device__ __forceinline__ void store_levels(int16_t *dst, const int16_t *lev)
{
    uint4 a, b;
    a.x = (uint16_t)lev[0] | ((uint32_t)(uint16_t)lev[1] << 16);
    a.y = (uint16_t)lev[2] | ((uint32_t)(uint16_t)lev[3] << 16);
    a.z = (uint16_t)lev[4] | ((uint32_t)(uint16_t)lev[5] << 16);
    a.w = (uint16_t)lev[6] | ((uint32_t)(uint16_t)lev[7] << 16);
    b.x = (uint16_t)lev[8] | ((uint32_t)(uint16_t)lev[9] << 16);
    b.y = (uint16_t)lev[10] | ((uint32_t)(uint16_t)lev[11] << 16);
    b.z = (uint16_t)lev[12] | ((uint32_t)(uint16_t)lev[13] << 16);
    b.w = (uint16_t)lev[14] | ((uint32_t)(uint16_t)lev[15] << 16);
    ((uint4 *)dst)[0] = a;
    ((uint4 *)dst)[1] = b;
}

// Zig-zag scan index of raster position r of a 4x4 block: the inverse of h264_zigzag4x4.
__device__ __forceinline__ int inv_zigzag4x4(int r)
{
    const uint8_t izz[16] = {0, 1, 5, 6, 2, 4, 7, 12, 3, 8, 11, 13, 9, 10, 14, 15};
    return izz[r];
}

// Syntax records of chroma lanes 16..23 and lane 25, the same for inter and intra macroblocks: a chroma lane stores its
// block's AC levels, nnz and DC level, and the first lane of each plane the nnz of the plane's DC block; lane 25 clears
// the unused half of the chroma DC record.
__device__ __forceinline__ void store_chroma_syntax(int16_t *cf, uint8_t *nn, int lane, const int16_t *lev, int nz,
                                                    const ChromaOut &co)
{
    if (lane < 24) {
        const int c = (lane - 16) >> 2, cb = lane & 3;
        store_levels(cf + (18 + c * 4 + cb) * 16, lev);
        nn[NNZ_CB + c * 4 + cb] = (uint8_t)nz;
        cf[17 * 16 + c * 4 + cb] = (int16_t)co.zdc;
        if (cb == 0)
            nn[NNZ_CBDC + c] = (uint8_t)__popc(co.m_dc & (0xfu << (16 + 4 * c)));
    } else if (lane == 25) {
        *(uint4 *)(cf + 17 * 16 + 8) = make_uint4(0, 0, 0, 0);
    }
}

// Quantiser constants of one lane's 4x4 block of an inter macroblock (luma lanes: QP, chroma lanes: QPc), so that luma
// and chroma lanes run the transform / quantisation / reconstruction as one instruction stream.  Same arithmetic as
// quant_block / dequant_ac (h264_core.cuh).
struct LaneQuant {
    int mf[3], ls[3]; // by position class
    int f, qbits, mul, rnd, sr;
};
__device__ __forceinline__ LaneQuant lane_quant_inter(int q)
{
    LaneQuant k;
    const int m = q % 6, e = q / 6;
#pragma unroll
    for (int c = 0; c < 3; c++) {
        k.mf[c] = h264_quant_mf[m][c];
        k.ls[c] = 16 * h264_dequant_v[m][c];
    }
    k.qbits = 15 + e;
    k.f = (1 << k.qbits) / 6;
    k.mul = e >= 4 ? 1 << (e - 4) : 1; // dequant_ac: (c * ls) * 2^(e - 4), or (c * ls + 2^(3 - e)) >> (4 - e)
    k.rnd = e >= 4 ? 0 : 1 << (3 - e);
    k.sr = e >= 4 ? 0 : 4 - e;
    return k;
}

// ================================================================================================
// K3 inter macroblock: integer luma MC, bilinear chroma MC (xFrac, yFrac in {0, 4}), 4x4 transform,
// quantisation, CBP, dequantisation, inverse transform, reconstruction (before deblocking).
// One warp per macroblock: lanes 0..15 luma 4x4 blocks, 16..23 chroma, 24/25 clear unused levels.
// All macroblocks of all lanes in parallel.  HBM / L2 bound.
// ================================================================================================
__global__ void __launch_bounds__(128) inter_kernel(Geom g, Step s, const uint8_t *__restrict__ src,
                                                    const uint8_t *__restrict__ ref, uint8_t *__restrict__ unf,
                                                    MbInfo *__restrict__ mbi, uint8_t *__restrict__ nnz,
                                                    int16_t *__restrict__ coef)
{
    if (lane_frame(s, blockIdx.y) < 0)
        return;
    const int lane = threadIdx.x & 31;
    const int mb = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (mb >= g.nmb)
        return;
    const int mbx = mb % g.mbw, mby = mb / g.mbw;
    const size_t fo = (size_t)blockIdx.y * g.frame_bytes;
    const size_t rec = (size_t)blockIdx.y * g.nmb + mb;
    const MbInfo me = mbi[rec];
    const bool luma = lane < 16, chroma = lane >= 16 && lane < 24;
    const int qp = g.qp, qpc = g.qpc;

    int pred[16], w[16], d[16];
    int16_t lev[16];
    int nz = 0;
    size_t out_off = 0;
    int out_stride = 0;
#pragma unroll
    for (int i = 0; i < 16; i++)
        d[i] = 0, pred[i] = 0;
    if (luma || chroma) {
        // One prediction fetch for luma and chroma lanes: every lane describes its 4x4 block by plane offset, plane size
        // and vector (luma: integer-pel, no fraction; chroma: mv / 8 with a fraction of 0 or 4 eighths, because the luma
        // vectors are integer-pel) and reads the 5 x 5 reference samples the bilinear filter can touch, per row as two
        // words: samples 0..3 (wa) and 1..4 (wb).
        const int c = (lane - 16) >> 2, cb = lane & 3;
        const size_t po = luma ? fo : fo + (size_t)g.W * g.H + (size_t)c * g.CW * g.CH;
        const int pw_ = luma ? g.W : g.CW, ph_ = luma ? g.H : g.CH;
        const int px = luma ? mbx * 16 + blk_x(lane) * 4 : mbx * 8 + (cb & 1) * 4;
        const int py = luma ? mby * 16 + blk_y(lane) * 4 : mby * 8 + (cb >> 1) * 4;
        const int mvx = me.mv[0], mvy = me.mv[1];
        const int rx = px + (luma ? mvx >> 2 : mvx >> 3), ry = py + (luma ? mvy >> 2 : mvy >> 3);
        const int xf = luma ? 0 : mvx & 7, yf = luma ? 0 : mvy & 7;
        const uint8_t *sp = src + po + (size_t)py * pw_ + px;
        const uint8_t *rp = ref + po;
        uint32_t wa[5], wb[5];
        if (rx >= 0 && rx + 7 < pw_ && ry >= 0 && ry + 4 < ph_) {
#pragma unroll
            for (int y = 0; y < 5; y++) {
                const uintptr_t a = (uintptr_t)(rp + (size_t)(ry + y) * pw_ + rx);
                const uint32_t *aw = (const uint32_t *)(a & ~(uintptr_t)3);
                const uint32_t lo = aw[0], hi = aw[1], sh = (uint32_t)(a & 3) * 8;
                wa[y] = __funnelshift_r(lo, hi, sh);
                wb[y] = __funnelshift_rc(lo, hi, sh + 8); // clamped: a shift of 32 is the high word
            }
        } else {
#pragma unroll
            for (int y = 0; y < 5; y++) {
                const uint8_t *rr = rp + (size_t)clip3_(0, ph_ - 1, ry + y) * pw_;
                uint32_t s5[5];
#pragma unroll
                for (int x = 0; x < 5; x++)
                    s5[x] = rr[clip3_(0, pw_ - 1, rx + x)];
                wa[y] = s5[0] | (s5[1] << 8) | (s5[2] << 16) | (s5[3] << 24);
                wb[y] = s5[1] | (s5[2] << 8) | (s5[3] << 16) | (s5[4] << 24);
            }
        }
        // ((8-xf)(8-yf) A + xf (8-yf) B + (8-xf) yf C + xf yf D + 32) >> 6 with xf, yf in {0, 4} is A, a rounding
        // average of two samples, or (A + B + C + D + 2) >> 2: four samples at a time on packed bytes.
#pragma unroll
        for (int y = 0; y < 4; y++) {
            const uint32_t sv = *(const uint32_t *)(sp + (size_t)y * pw_);
            uint32_t pw;
            if (xf == 0 && yf == 0)
                pw = wa[y];
            else if (yf == 0)
                pw = __vavgu4(wa[y], wb[y]);
            else if (xf == 0)
                pw = __vavgu4(wa[y], wa[y + 1]);
            else {
                const uint32_t m = 0x00ff00ffu;
                const uint32_t ev = (wa[y] & m) + (wb[y] & m) + (wa[y + 1] & m) + (wb[y + 1] & m) + 0x00020002u;
                const uint32_t od =
                    ((wa[y] >> 8) & m) + ((wb[y] >> 8) & m) + ((wa[y + 1] >> 8) & m) + ((wb[y + 1] >> 8) & m) + 0x00020002u;
                pw = ((ev >> 2) & m) | (((od >> 2) & m) << 8);
            }
#pragma unroll
            for (int x = 0; x < 4; x++) {
                const int p = (int)((pw >> (8 * x)) & 0xff);
                pred[y * 4 + x] = p;
                d[y * 4 + x] = (int)((sv >> (8 * x)) & 0xff) - p;
            }
        }
        out_off = po + (size_t)py * pw_ + px;
        out_stride = pw_;
    }
    // transform and quantisation, luma and chroma lanes together (idle lanes carry zeros); the chroma DC goes its own way
    const LaneQuant lq = lane_quant_inter(luma ? qp : qpc);
    fdct4x4(d, w);
#pragma unroll
    for (int i = 0; i < 16; i++) {
        const int r = h264_zigzag4x4[i];
        int z = quant1(w[r], lq.mf[pos_class(r)], lq.f, lq.qbits);
        if (i == 0 && chroma)
            z = 0;
        lev[i] = (int16_t)z;
        nz += z != 0;
    }
    ChromaOut co = chroma_dc_path(w, nz, chroma, lane, qpc, 0);
    unsigned m_l = __ballot_sync(0xffffffffu, luma && nz > 0);
    int cbpl = ((m_l & 0x000f) ? 1 : 0) | ((m_l & 0x00f0) ? 2 : 0) | ((m_l & 0x0f00) ? 4 : 0) | ((m_l & 0xf000) ? 8 : 0);

    // levels that are not coded (chroma AC without cbp 2) do not reach the reconstruction
    const bool coded = luma ? nz != 0 : (chroma && co.cbpc == 2);
    // most macroblocks of a well-predicted picture have no residual at all: their reconstruction is the prediction
    const bool any_residual = __any_sync(0xffffffffu, coded || (chroma && co.cbpc != 0));
    if (luma || chroma) {
        uint8_t *op = unf + out_off;
        if (any_residual) {
            int r[16];
#pragma unroll
            for (int i = 0; i < 16; i++) {
                const int rr = h264_zigzag4x4[i];
                d[rr] = coded ? ((int)lev[i] * lq.ls[pos_class(rr)] * lq.mul + lq.rnd) >> lq.sr : 0;
            }
            if (chroma)
                d[0] = co.cbpc ? co.dcq : 0;
            idct4x4(d, r);
#pragma unroll
            for (int y = 0; y < 4; y++) {
                int v[4];
#pragma unroll
                for (int x = 0; x < 4; x++)
                    v[x] = clip255_(pred[y * 4 + x] + r[y * 4 + x]);
                *(uint32_t *)(op + (size_t)y * out_stride) = pack4(v);
            }
        } else {
#pragma unroll
            for (int y = 0; y < 4; y++)
                *(uint32_t *)(op + (size_t)y * out_stride) = pack4(pred + 4 * y);
        }
    }
    // syntax records
    int16_t *cf = coef + rec * COEF_STRIDE;
    uint8_t *nn = nnz + rec * NNZ_STRIDE;
    if (luma) {
        store_levels(cf + lane * 16, lev);
        nn[lane] = (uint8_t)nz;
    } else if (lane == 24) {
        store_levels(cf + 16 * 16, lev); // zeros: no Intra16x16 DC block
        nn[NNZ_DC16] = 0;
    } else
        store_chroma_syntax(cf, nn, lane, lev, nz, co);
    if (lane == 0) {
        MbInfo m = me;
        m.type = MB_P16x16;
        m.cbp = (uint8_t)(cbpl | (co.cbpc << 4));
        mbi[rec] = m;
    }
}

// ================================================================================================
// K2 median MV prediction, mvd and the P_Skip decision.  One thread per macroblock (called from bs_kernel); runs
// after all MVs of the frame are final (they never change here), so it is order independent.
// ================================================================================================
__device__ __forceinline__ void mvp_skip_mb(const Geom &g, MbInfo *frame, int mb)
{
    MbInfo m = frame[mb];
    if (m.type != MB_P16x16 && m.type != MB_PSKIP)
        return;
    int mvp[2], smv[2];
    predict_mv(frame, g.mbw, g.srows, mb % g.mbw, mb / g.mbw, mvp, smv);
    int16_t mvdx = (int16_t)(m.mv[0] - mvp[0]), mvdy = (int16_t)(m.mv[1] - mvp[1]);
    uint8_t type = MB_P16x16;
    if (m.cbp == 0 && m.mv[0] == smv[0] && m.mv[1] == smv[1]) {
        type = MB_PSKIP;
        mvdx = mvdy = 0;
    }
    // only fields nobody else reads in this kernel are written (type is read, but P16x16 and PSKIP
    // are treated alike by predict_mv)
    frame[mb].mvd[0] = mvdx;
    frame[mb].mvd[1] = mvdy;
    frame[mb].type = type;
}


// ================================================================================================
// K4 intra macroblocks of I frames: Intra16x16 (V/H/DC/Plane) + chroma (DC/H/V/Plane), mode by SAD,
// transform / quant / recon.  Neighbours are the UNFILTERED reconstruction, so macroblock (x, y)
// depends on (x-1, y) and on row y-1 up to x: one warp walks one macroblock row and publishes its
// progress; the row below spins on it (wavefront).  INTRA_ROWS consecutive rows share a CTA: between them the
// progress counter is a shared-memory word (a hop of a few hundred cycles; the pixels themselves go through L2),
// only every INTRA_ROWS-th row synchronises through flags[row] in global memory (a hop of ~10^4 cycles).  Lanes as
// in K3.  Bound: dependency latency (mbw + mbh steps per frame) -- many lanes run side by side.
// ================================================================================================
// p_intra extension, decision (oracle: p_intra_decide): one warp per macroblock, all macroblocks in parallel.  Best
// Intra16x16 SAD against the neighbours as they are after the all-inter reconstruction of the picture (inter_kernel),
// chosen when sad16 + 8 * lambda < the motion search's best cost (MbInfo::pad).  The chosen macroblocks are then
// re-coded by intra_kernel in wavefront order.
__global__ void __launch_bounds__(128) pintra_decide_kernel(Geom g, Step s, const uint8_t *__restrict__ src,
                                                           const uint8_t *__restrict__ unf, const MbInfo *__restrict__ mbi,
                                                           uint8_t *__restrict__ want, int *__restrict__ count)
{
    if (lane_frame(s, blockIdx.y) < 0)
        return;
    __shared__ uint8_t top_s[4][20], left_s[4][16];
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5, mb = blockIdx.x * 4 + wrp;
    if (mb >= g.nmb)
        return;
    const int mbx = mb % g.mbw, mby = mb / g.mbw, has_top = (mby % g.srows) != 0, has_left = mbx > 0;
    const size_t fo = (size_t)blockIdx.y * g.frame_bytes, rec = (size_t)blockIdx.y * g.nmb + mb;
    const uint8_t *dst = unf + fo + (size_t)(mby * 16) * g.W + mbx * 16;
    uint8_t *top = top_s[wrp], *left = left_s[wrp];
    if (lane < 17)
        top[lane] = (has_top && (lane > 0 || has_left)) ? dst[-g.W - 1 + lane] : 0;
    if (lane >= 16)
        left[lane - 16] = has_left ? dst[(size_t)(lane - 16) * g.W - 1] : 0;
    __syncwarp();
    const bool luma = lane < 16;
    const int bx = blk_x(lane & 15) * 4, by = blk_y(lane & 15) * 4;
    uint32_t sv[4] = {0, 0, 0, 0};
    if (luma)
#pragma unroll
        for (int y = 0; y < 4; y++)
            sv[y] = *(const uint32_t *)(src + fo + (size_t)(mby * 16 + by + y) * g.W + mbx * 16 + bx);
    uint32_t best = 0xffffffffu;
#pragma unroll 1
    for (int mode = 0; mode < 4; mode++) {
        const bool avail = !((mode == 0 && !has_top) || (mode == 1 && !has_left) || (mode == 3 && !(has_top && has_left)));
        int sad = 0;
        if (avail && luma) {
            int p[16];
            pred16_block(mode, top, left, has_top, has_left, bx, by, p);
#pragma unroll
            for (int i = 0; i < 16; i++)
                sad += iabs_((int)((sv[i >> 2] >> (8 * (i & 3))) & 0xff) - p[i]);
        }
#pragma unroll
        for (int o = 8; o >= 1; o >>= 1)
            sad += __shfl_xor_sync(0xffffffffu, sad, o);
        if (avail && (uint32_t)sad < best)
            best = (uint32_t)sad;
    }
    if (lane == 0) {
        const bool w = best + 8u * (uint32_t)g.lambda < mbi[rec].pad;
        want[rec] = (uint8_t)w;
        if (w)
            atomicAdd(count + blockIdx.y, 1);
    }
}

#define INTRA_ROWS 8

// Per-warp shared state of the Intra4x4 trial (intra4x4 extension).
struct __align__(16) I4Work {
    uint8_t patch[17][24]; // row 0: samples above (col 3 above-left, 4..19 above, 20..23 above-right); rows 1..16: col 3 =
                           // left neighbours, cols 4..19 = the macroblock as it is reconstructed block by block
    uint8_t nb[16];        // neighbours of the current block: 0..7 above / above-right, 8..11 left, 12 above-left
    uint8_t mode[16], nnzb[16]; // per luma4x4BlkIdx
    uint8_t left_mode[16]; // modes of the macroblock to the left
    uint8_t left_is_i4;
};

// Tries to code the macroblock's luma as Intra4x4 (oracle: try_intra4x4): block by block, mode = argmin over the
// available modes of (SAD + lambda * modebits) << 4 | mode (modebits 1 for the predicted mode, 4 otherwise); the block
// is reconstructed at once because the next blocks predict from it.  Gives up as soon as the accumulated cost reaches
// cost16.  Warp-collective: lane = sample (x, y) of the current block in both half-warps, the halves evaluate two
// modes at a time; transforms run across the 16 lanes with shuffles.  top_kind: -1 no macroblock above, 0 it is not
// Intra4x4, 1 its modes are at top_modes.
__device__ __forceinline__ bool intra4x4_trial(const Geom &g, I4Work &w, int lane, const uint32_t *sv, bool has_topmb,
                                               bool has_leftmb, bool has_trmb, int top_kind, const uint8_t *top_modes,
                                               uint32_t cost16, int16_t *cf, int &cbp_out)
{
    const int r = lane & 15, x = r & 3, y = r >> 2, half = lane & 16, qp = g.qp;
    const int qbits = 15 + qp / 6, f = (1 << qbits) / 3, cls = pos_class(r);
    uint32_t cost4 = 0;
    int cbp = 0;
    for (int b = 0; b < 16; b++) {
        const int bx = blk_x(b), by = blk_y(b);
        const bool ht = by > 0 || has_topmb, hl = bx > 0 || has_leftmb, htl = ht && hl;
        const bool htr = by == 0 ? (has_topmb && (bx < 3 || has_trmb)) : (bx < 3 && xy2blk(bx + 1, by - 1) < b);
        if (lane < 8)
            w.nb[lane] = ht ? w.patch[by * 4][4 + bx * 4 + ((lane < 4 || htr) ? lane : 3)] : 0;
        else if (lane < 12)
            w.nb[lane] = hl ? w.patch[1 + by * 4 + (lane - 8)][3 + bx * 4] : 0;
        else if (lane == 12)
            w.nb[12] = htl ? w.patch[by * 4][3 + bx * 4] : 0;
        __syncwarp();
        int ma, mb2; // modes of the blocks to the left / above, for the predicted mode
        if (bx > 0)
            ma = w.mode[xy2blk(bx - 1, by)];
        else
            ma = !has_leftmb ? -1 : (w.left_is_i4 ? (int)w.left_mode[xy2blk(3, by)] : 2);
        if (by > 0)
            mb2 = w.mode[xy2blk(bx, by - 1)];
        else
            mb2 = top_kind < 0 ? -1 : (top_kind == 0 ? 2 : (int)__ldcg(top_modes + xy2blk(bx, 3)));
        const int pm = (ma < 0 || mb2 < 0) ? 2 : imin_(ma, mb2);
        // source sample (x, y) of block b: lane b holds the block's four rows
        const uint32_t r0 = __shfl_sync(0xffffffffu, sv[0], b), r1 = __shfl_sync(0xffffffffu, sv[1], b);
        const uint32_t r2 = __shfl_sync(0xffffffffu, sv[2], b), r3 = __shfl_sync(0xffffffffu, sv[3], b);
        const int sp = (int)(((y & 2 ? (y & 1 ? r3 : r2) : (y & 1 ? r1 : r0)) >> (8 * x)) & 0xff);
        const int m = w.nb[12];
        uint32_t best = 0xffffffffu;
#pragma unroll 1
        for (int i = 0; i < 5; i++) {
            const int mode = 2 * i + (half >> 4);
            const bool need_top = mode == 0 || mode == 3 || mode == 7 || (mode >= 4 && mode <= 6);
            const bool need_left = mode == 1 || mode == 8 || (mode >= 4 && mode <= 6);
            const bool valid = mode <= 8 && (!need_top || ht) && (!need_left || hl) && (!(mode >= 4 && mode <= 6) || htl);
            int ad = 0;
            if (valid)
                ad = iabs_(sp - pred4x4_pixel(mode, x, y, w.nb, w.nb + 8, m, ht, hl));
#pragma unroll
            for (int o = 8; o >= 1; o >>= 1)
                ad += __shfl_xor_sync(0xffffffffu, ad, o);
            const uint32_t key = valid ? (((uint32_t)ad + (uint32_t)(g.lambda * (mode == pm ? 1 : 4))) << 4) | (uint32_t)mode : 0xffffffffu;
            best = key < best ? key : best;
        }
        {
            const uint32_t o = __shfl_xor_sync(0xffffffffu, best, 16);
            best = o < best ? o : best;
        }
        cost4 += best >> 4;
        if (cost4 >= cost16)
            return false;
        const int mode_b = (int)(best & 15);
        // ---- reconstruct the block: residual, 4x4 transform, quantisation, and back ----
        const int pv = pred4x4_pixel(mode_b, x, y, w.nb, w.nb + 8, m, ht, hl);
        int v = sp - pv;
        {
            const int rb = lane & ~3; // forward transform, rows
            const int a = __shfl_sync(0xffffffffu, v, rb), b1 = __shfl_sync(0xffffffffu, v, rb + 1);
            const int c = __shfl_sync(0xffffffffu, v, rb + 2), e = __shfl_sync(0xffffffffu, v, rb + 3);
            const int s03 = a + e, d03 = a - e, s12 = b1 + c, d12 = b1 - c;
            v = x == 0 ? s03 + s12 : (x == 1 ? 2 * d03 + d12 : (x == 2 ? s03 - s12 : d03 - 2 * d12));
        }
        {
            const int cbase = half + x; // columns
            const int a = __shfl_sync(0xffffffffu, v, cbase), b1 = __shfl_sync(0xffffffffu, v, cbase + 4);
            const int c = __shfl_sync(0xffffffffu, v, cbase + 8), e = __shfl_sync(0xffffffffu, v, cbase + 12);
            const int s03 = a + e, d03 = a - e, s12 = b1 + c, d12 = b1 - c;
            v = y == 0 ? s03 + s12 : (y == 1 ? 2 * d03 + d12 : (y == 2 ? s03 - s12 : d03 - 2 * d12));
        }
        const int z = quant1(v, h264_quant_mf[qp % 6][cls], f, qbits);
        const int n = __popc(__ballot_sync(0xffffffffu, z != 0) & 0xffffu);
        if (lane < 16)
            cf[b * 16 + inv_zigzag4x4(r)] = (int16_t)z;
        v = n ? dequant_ac(z, qp, cls) : 0;
        {
            const int rb = lane & ~3; // inverse transform, rows
            const int d0 = __shfl_sync(0xffffffffu, v, rb), d1 = __shfl_sync(0xffffffffu, v, rb + 1);
            const int d2 = __shfl_sync(0xffffffffu, v, rb + 2), d3 = __shfl_sync(0xffffffffu, v, rb + 3);
            const int e0 = d0 + d2, e1 = d0 - d2, e2 = (d1 >> 1) - d3, e3 = d1 + (d3 >> 1);
            v = x == 0 ? e0 + e3 : (x == 1 ? e1 + e2 : (x == 2 ? e1 - e2 : e0 - e3));
        }
        {
            const int cbase = half + x; // columns
            const int d0 = __shfl_sync(0xffffffffu, v, cbase), d1 = __shfl_sync(0xffffffffu, v, cbase + 4);
            const int d2 = __shfl_sync(0xffffffffu, v, cbase + 8), d3 = __shfl_sync(0xffffffffu, v, cbase + 12);
            const int e0 = d0 + d2, e1 = d0 - d2, e2 = (d1 >> 1) - d3, e3 = d1 + (d3 >> 1);
            v = ((y == 0 ? e0 + e3 : (y == 1 ? e1 + e2 : (y == 2 ? e1 - e2 : e0 - e3))) + 32) >> 6;
        }
        if (lane < 16)
            w.patch[1 + by * 4 + y][4 + bx * 4 + x] = (uint8_t)clip255_(pv + v);
        if (lane == 0) {
            w.mode[b] = (uint8_t)mode_b;
            w.nnzb[b] = (uint8_t)n;
        }
        if (n)
            cbp |= 1 << (b >> 2);
        __syncwarp();
    }
    cbp_out = cbp;
    return true;
}
__global__ void __launch_bounds__(INTRA_ROWS * 32) intra_kernel(Geom g, Step s, const uint8_t *__restrict__ src,
                                                                uint8_t *unf, MbInfo *__restrict__ mbi,
                                                                uint8_t *__restrict__ nnz, int16_t *__restrict__ coef,
                                                                int *flags, uint8_t *i4, const uint8_t *pwant,
                                                                const int *pcount)
{
    // pwant != null: P frame of the p_intra extension -- only the macroblocks marked by pintra_decide_kernel are coded
    // (as Intra16x16, over their inter version); the wavefront still runs over all of them because a marked macroblock
    // predicts from whatever its neighbours ended up as.
    if (lane_frame(s, blockIdx.y) < 0 || (pwant && pcount[blockIdx.y] == 0))
        return;
    __shared__ I4Work i4w_s[INTRA_ROWS];
    __shared__ uint8_t topY_s[INTRA_ROWS][20], leftY_s[INTRA_ROWS][16], topC_s[INTRA_ROWS][2][12], leftC_s[INTRA_ROWS][2][8];
    __shared__ volatile int progress[INTRA_ROWS]; // macroblocks finished by each row of this CTA
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5, row = blockIdx.x * INTRA_ROWS + wrp;
    if (threadIdx.x < INTRA_ROWS)
        progress[threadIdx.x] = 0;
    __syncthreads();
    if (row >= g.mbh)
        return;
    uint8_t *topY = topY_s[wrp], *leftY = leftY_s[wrp];
    uint8_t(*topC)[12] = topC_s[wrp];
    uint8_t(*leftC)[8] = leftC_s[wrp];
    I4Work &i4w = i4w_s[wrp];
    if (lane == 0)
        i4w.left_is_i4 = 0;
    const size_t fo = (size_t)blockIdx.y * g.frame_bytes;
    int *fl = flags + (size_t)blockIdx.y * g.mbh;
    const bool luma = lane < 16, chroma = lane >= 16 && lane < 24;
    const int qp = g.qp, qpc = g.qpc;
    const int c = (lane - 16) >> 2, cb = lane & 3;
    const int bx = luma ? blk_x(lane) * 4 : (cb & 1) * 4, by = luma ? blk_y(lane) * 4 : (cb >> 1) * 4;
    const size_t plane_off = luma ? fo : fo + (size_t)g.W * g.H + (size_t)(chroma ? c : 0) * g.CW * g.CH;
    const int stride = luma ? g.W : g.CW, mbsz = luma ? 16 : 8;

    // Row `row` has finished macroblocks [0, n).  The CTA's last row releases its global flag, which the first row of the
    // next CTA reads; the other rows fence their pixels (global stores, read back through L2 by the row below) before
    // raising the shared counter.
    auto publish = [&](int n) {
        if (lane == 0) {
            if (wrp == INTRA_ROWS - 1 || row == g.mbh - 1)
                st_release(fl + row, n);
            else {
                __threadfence();
                progress[wrp] = n;
            }
        }
    };

    const bool try_i4 = g.intra4x4 && !pwant;
    for (int mbx = 0; mbx < g.mbw; mbx++) {
        const int has_top = (row % g.srows) != 0, has_left = mbx > 0; // the row above may belong to another slice
        const size_t rec = (size_t)blockIdx.y * g.nmb + (size_t)row * g.mbw + mbx;
        if (pwant) {
            if (!pwant[rec]) { // stays inter: nothing to do but to let the row below pass
                publish(mbx + 1);
                continue;
            }
            if (has_left) { // the left neighbour may be an inter macroblock: its column comes from the picture, not from this warp
                const uint8_t *ly = unf + fo + (size_t)(row * 16) * g.W + mbx * 16 - 1;
                if (lane < 16)
                    leftY[lane] = __ldcg(ly + (size_t)lane * g.W);
                else {
                    const int pl = (lane - 16) >> 3, i = lane & 7;
                    leftC[pl][i] = __ldcg(unf + fo + (size_t)g.W * g.H + (size_t)pl * g.CW * g.CH + (size_t)(row * 8 + i) * g.CW + mbx * 8 - 1);
                }
            }
        }
        // source block (independent of the wavefront)
        uint32_t sv[4] = {0, 0, 0, 0};
        const size_t blk_off = plane_off + (size_t)(row * mbsz + by) * stride + mbx * mbsz + bx;
        if (luma || chroma) {
#pragma unroll
            for (int y = 0; y < 4; y++)
                sv[y] = *(const uint32_t *)(src + blk_off + (size_t)y * stride);
        }
        if (has_top) {
            if (lane == 0) {
                // Intra4x4 predicts from the macroblock above and to the right as well
                const int need = try_i4 ? imin_(mbx + 2, g.mbw) : mbx + 1;
                if (wrp > 0) { // the row above lives in this CTA
                    while (progress[wrp - 1] < need)
                        __nanosleep(20);
                    __threadfence_block();
                } else
                    while (ld_acquire(fl + row - 1) < need)
                        ;
            }
            __syncwarp();
            const uint8_t *ty = unf + fo + (size_t)(row * 16 - 1) * g.W + mbx * 16 - 1;
            if (lane < 17 && (lane > 0 || has_left))
                topY[lane] = __ldcg(ty + lane);
            if (try_i4 && lane >= 17 && lane < 21 && mbx + 1 < g.mbw)
                i4w.patch[0][20 + lane - 17] = __ldcg(ty + lane); // above-right
            if (lane < 9 || (lane >= 16 && lane < 25)) {
                int pl = lane >> 4, i = lane & 15;
                const uint8_t *tc = unf + fo + (size_t)g.W * g.H + (size_t)pl * g.CW * g.CH +
                                    (size_t)(row * 8 - 1) * g.CW + mbx * 8 - 1;
                if (i > 0 || has_left)
                    topC[pl][i] = __ldcg(tc + i);
            }
        }
        __syncwarp();

        // ---- mode decision: SAD of every available mode, summed over the 16-lane group ----
        const uint8_t *tp = luma ? topY : topC[chroma ? c : 0];
        const uint8_t *lp = luma ? leftY : leftC[chroma ? c : 0];
        uint32_t best = 0xffffffffu;
#pragma unroll 1
        for (int mode = 0; mode < 4; mode++) {
            // luma: 0 V 1 H 2 DC 3 P ; chroma: 0 DC 1 H 2 V 3 P  (availability per group)
            int need_top = luma ? (mode == 0 || mode == 3) : (mode == 2 || mode == 3);
            int need_left = (mode == 1 || mode == 3);
            bool avail = (!need_top || has_top) && (!need_left || has_left);
            int sad = 0;
            if (avail && (luma || chroma)) {
                int p[16];
                if (luma)
                    pred16_block(mode, tp, lp, has_top, has_left, bx, by, p);
                else
                    predc_block(mode, tp, lp, has_top, has_left, bx, by, p);
#pragma unroll
                for (int i = 0; i < 16; i++)
                    sad += iabs_((int)((sv[i >> 2] >> (8 * (i & 3))) & 0xff) - p[i]);
            }
#pragma unroll
            for (int o = 8; o >= 1; o >>= 1)
                sad += __shfl_xor_sync(0xffffffffu, sad, o);
            uint32_t key = avail ? (((uint32_t)sad << 2) | (uint32_t)mode) : 0xffffffffu;
            best = key < best ? key : best;
        }
        const int mode = (int)(best & 3);
        // ---- intra4x4 extension: try Intra4x4 against the best Intra16x16 cost (luma only; chroma is unchanged) ----
        bool use_i4 = false;
        int cbp4 = 0;
        if (try_i4) {
            if (lane < 17)
                i4w.patch[0][3 + lane] = (has_top && (lane > 0 || has_left)) ? topY[lane] : 0;
            if (lane < 16)
                i4w.patch[1 + lane][3] = has_left ? leftY[lane] : 0;
            __syncwarp();
            int top_kind = -1;
            if (has_top)
                top_kind = __ldcg((const uint8_t *)(mbi + rec - g.mbw)) == MB_I4x4; // MbInfo::type is the first byte
            use_i4 = intra4x4_trial(g, i4w, lane, sv, has_top, has_left, mbx + 1 < g.mbw, top_kind, i4 + (rec - g.mbw) * 16,
                                    __shfl_sync(0xffffffffu, best, 0) >> 2, coef + rec * COEF_STRIDE, cbp4);
        }
        const bool luma16 = luma && !use_i4; // lanes that code an Intra16x16 luma block
        int pred[16], d[16], w[16];
        int16_t lev[16];
        int nz = 0;
#pragma unroll
        for (int i = 0; i < 16; i++)
            pred[i] = 0, w[i] = 0, lev[i] = 0;
        if (luma16 || chroma) {
            if (luma)
                pred16_block(mode, tp, lp, has_top, has_left, bx, by, pred);
            else
                predc_block(mode, tp, lp, has_top, has_left, bx, by, pred);
#pragma unroll
            for (int i = 0; i < 16; i++)
                d[i] = (int)((sv[i >> 2] >> (8 * (i & 3))) & 0xff) - pred[i];
            fdct4x4(d, w);
            nz = quant_block(w, luma ? qp : qpc, 1, 1, lev);
        }
        // ---- Intra16x16 DC: 4x4 Hadamard across the 16 luma lanes ----
        int D[16], Y[16];
#pragma unroll
        for (int p = 0; p < 16; p++)
            D[p] = __shfl_sync(0xffffffffu, w[0], xy2blk(p & 3, p >> 2));
        hadamard4x4(D, Y);
        int qbits = 15 + qp / 6, f = (1 << qbits) / 3;
        int ydc = 0;
#pragma unroll
        for (int p = 0; p < 16; p++)
            ydc = (lane == p) ? Y[p] : ydc;
        int zdc16 = luma16 ? quant1(ydc, h264_quant_mf[qp % 6][0], 4 * f, qbits + 2) : 0; // raster position = lane
        unsigned m_dc16 = __ballot_sync(0xffffffffu, zdc16 != 0);
#pragma unroll
        for (int p = 0; p < 16; p++)
            D[p] = __shfl_sync(0xffffffffu, zdc16, p);
        hadamard4x4(D, Y);
        int fdc = 0;
        {
            int mypos = blk_y(lane & 15) * 4 + blk_x(lane & 15);
#pragma unroll
            for (int p = 0; p < 16; p++)
                fdc = (mypos == p) ? Y[p] : fdc;
        }
        unsigned m_ac = __ballot_sync(0xffffffffu, luma16 && nz > 0);
        const int any_ac = m_ac != 0;
        ChromaOut co = chroma_dc_path(w, nz, chroma, lane, qpc, 1);

        // ---- reconstruction ----
        int recv[16];
        if (luma && use_i4) { // the Intra4x4 reconstruction is in the trial's patch
            uint8_t *op = unf + blk_off;
#pragma unroll
            for (int y = 0; y < 4; y++) {
                const uint32_t v = *(const uint32_t *)&i4w.patch[1 + by + y][4 + bx];
                *(uint32_t *)(op + (size_t)y * stride) = v;
                recv[y * 4 + 3] = (int)(v >> 24);
            }
        }
        if (luma16 || chroma) {
            int dd[16], r[16];
#pragma unroll
            for (int i = 0; i < 16; i++)
                dd[i] = 0;
            if (luma) {
                if (any_ac)
                    dequant_block(lev, qp, 1, dd);
                dd[0] = dequant_luma_dc(fdc, qp);
            } else {
                if (co.cbpc == 2)
                    dequant_block(lev, qpc, 1, dd);
                dd[0] = co.cbpc ? co.dcq : 0;
            }
            idct4x4(dd, r);
#pragma unroll
            for (int i = 0; i < 16; i++)
                recv[i] = clip255_(pred[i] + r[i]);
            uint8_t *op = unf + blk_off;
#pragma unroll
            for (int y = 0; y < 4; y++)
                *(uint32_t *)(op + (size_t)y * stride) = pack4(recv + y * 4);
        }
        __syncwarp(); // everybody is done reading top/left of this macroblock
        if (luma && bx == 12) {
#pragma unroll
            for (int y = 0; y < 4; y++)
                leftY[by + y] = (uint8_t)recv[y * 4 + 3];
        }
        if (chroma && bx == 4) {
#pragma unroll
            for (int y = 0; y < 4; y++)
                leftC[c][by + y] = (uint8_t)recv[y * 4 + 3];
        }
        // ---- syntax records ----
        int16_t *cf = coef + rec * COEF_STRIDE;
        uint8_t *nn = nnz + rec * NNZ_STRIDE;
        if (luma && use_i4) { // the levels were stored by the trial
            nn[lane] = i4w.nnzb[lane];
            cf[16 * 16 + inv_zigzag4x4(lane)] = 0;
            i4[rec * 16 + lane] = i4w.mode[lane];
            i4w.left_mode[lane] = i4w.mode[lane];
        } else if (luma) {
            store_levels(cf + lane * 16, lev);
            nn[lane] = (uint8_t)(any_ac ? nz : 0);
            cf[16 * 16 + inv_zigzag4x4(lane)] = (int16_t)zdc16;
            if (g.intra4x4)
                i4[rec * 16 + lane] = 0;
        } else if (lane == 24) {
            nn[NNZ_DC16] = (uint8_t)__popc(m_dc16 & 0xffffu);
        } else
            store_chroma_syntax(cf, nn, lane, lev, nz, co);
        int cmode = __shfl_sync(0xffffffffu, mode, 16);
        if (lane == 0) {
            MbInfo m;
            m.type = use_i4 ? MB_I4x4 : MB_I16x16;
            m.i16_mode = (uint8_t)(use_i4 ? 0 : mode);
            m.chroma_mode = (uint8_t)cmode;
            m.cbp = (uint8_t)((use_i4 ? cbp4 : (any_ac ? 15 : 0)) | (co.cbpc << 4));
            i4w.left_is_i4 = (uint8_t)use_i4;
            m.mv[0] = m.mv[1] = m.mvd[0] = m.mvd[1] = 0;
            m.pad = 0;
            mbi[rec] = m;
        }
        __syncwarp();
        publish(mbx + 1);
    }
}

// ================================================================================================
// K5 in-loop deblocking filter (H.264 8.7; slice offsets 0, cedar.c:1024-1029).
//
// bs_kernel: boundary strengths of all 32 edge segments of every macroblock, fully parallel
// (record = [dir][edge][segment] bytes: dir 0 vertical edges, 1 horizontal).
//
// deblock_kernel: standard-exact macroblock raster order realised as a 1:1 wavefront: an iteration filters a macroblock's
// inner vertical edges, its horizontal edges and the LEFT edge of the next macroblock, after which the macroblock is final,
// so (x, y) only waits for (x, y-1) (the raster order itself would need (x+1, y-1): two steps of lag per row).  Luma and
// chroma run in separate CTAs with independent progress flags.  Reads the unfiltered frame `unf`, writes the reference
// frame `rec`.  The next macroblock's pixels and strengths are prefetched into registers before the current one waits on
// the row above.
// Bound: dependency latency (mbw + mbh - 1 steps per frame).
// ================================================================================================
// with_mvp: the thread of edge (dir 0, e 0) also runs K2 (mvp_skip_mb) for its macroblock, which saves a launch on the
// critical chain.  K2 only rewrites type P16x16 -> PSKIP and mvd, neither of which a boundary strength depends on.
__global__ void bs_kernel(Geom g, Step s, MbInfo *mbi, const uint8_t *__restrict__ nnz, uint8_t *__restrict__ bs,
                          int with_mvp)
{
    if (lane_frame(s, blockIdx.y) < 0)
        return;
    int idx = blockIdx.x * blockDim.x + threadIdx.x; // (macroblock, dir, edge)
    int mb = idx >> 3, dir = (idx >> 2) & 1, e = idx & 3;
    if (mb >= g.nmb)
        return;
    const MbInfo *fm = mbi + (size_t)blockIdx.y * g.nmb;
    const uint8_t *fn = nnz + (size_t)blockIdx.y * g.nmb * NNZ_STRIDE;
    const int mbx = mb % g.mbw, mby = mb / g.mbw;
    const MbInfo cur = fm[mb];
    const uint8_t *ncur = fn + (size_t)mb * NNZ_STRIDE;
    uint32_t out = 0;
    if (e == 0) {
        bool avail = dir == 0 ? mbx > 0 : mby > 0;
        if (avail) {
            int nb = dir == 0 ? mb - 1 : mb - g.mbw;
            const MbInfo nbm = fm[nb];
            const uint8_t *nn = fn + (size_t)nb * NNZ_STRIDE;
#pragma unroll
            for (int sg = 0; sg < 4; sg++) {
                int bp = dir == 0 ? xy2blk(3, sg) : xy2blk(sg, 3), bq = dir == 0 ? xy2blk(0, sg) : xy2blk(sg, 0);
                out |= (uint32_t)boundary_strength(nbm, nn[bp], cur, ncur[bq], 1) << (8 * sg);
            }
        }
    } else {
#pragma unroll
        for (int sg = 0; sg < 4; sg++) {
            int bp = dir == 0 ? xy2blk(e - 1, sg) : xy2blk(sg, e - 1), bq = dir == 0 ? xy2blk(e, sg) : xy2blk(sg, e);
            out |= (uint32_t)boundary_strength(cur, ncur[bp], cur, ncur[bq], 0) << (8 * sg);
        }
    }
    ((uint32_t *)bs)[((size_t)blockIdx.y * g.nmb + mb) * 8 + dir * 4 + e] = out;
    if (with_mvp && dir == 0 && e == 0)
        mvp_skip_mb(g, mbi + (size_t)blockIdx.y * g.nmb, mb);
}

// Shared-memory mailbox between a filtering warp and its two helper warps.
struct DeblockMail {
    volatile int top_ready;    // loader -> main: top rows of macroblocks [0, top_ready) are in the ring
    volatile int top_consumed; // main -> loader: ring slots of macroblocks [0, top_consumed) are free again
    volatile int done;         // main -> publisher: macroblocks [0, done) are completely stored
};

__device__ __forceinline__ int ld_relaxed(const int *p)
{
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Loader warp: as soon as the row above has progressed far enough, fetches the top neighbour rows of the
// next macroblock from L2 into a 2-slot shared ring, so the filtering warp never waits on a global round
// trip.  `load_top(slot, mbx)` is executed by the whole warp.
template <class LoadTop>
__device__ __forceinline__ void deblock_loader(DeblockMail *mail, const int *fl_above, int mbw, int lane, LoadTop load_top)
{
    for (int x = 0; x < mbw; x++) {
        const int need = x + 1; // macroblock x of the row above is final once that row has finished its iteration x
        if (lane == 0) {
            while (mail->top_consumed + 2 <= x) // both ring slots still in use
                __nanosleep(64);
            while (ld_relaxed(fl_above) < need)
                __nanosleep(32);
            asm volatile("fence.acq_rel.gpu;" ::: "memory"); // acquire: the row above's pixels before its flag
        }
        __syncwarp();
        load_top(x & 1, x);
        __threadfence_block();
        __syncwarp();
        if (lane == 0)
            mail->top_ready = x + 1;
    }
}

// Publisher warp: publishes the filtering warp's progress with a gpu-scope release (the fence inside
// st.release covers the filtering warp's stores, observed through the shared `done` counter), so the
// filtering warp itself never stalls on a memory fence.
__device__ __forceinline__ void deblock_publisher(DeblockMail *mail, int *fl_mine, int mbw, int lane)
{
    if (lane != 0)
        return;
    int published = 0;
    while (published < mbw) {
        int d = mail->done;
        if (d > published) {
            __threadfence_block();
            st_release(fl_mine, d);
            published = d;
        } else
            __nanosleep(64);
    }
}

// One CTA filters `cta_rows` (<= DB_ROWS, chosen by the host so that the CTAs of a picture are equally tall: 68 rows = 4 x 17)
// consecutive macroblock rows of one plane type (blockIdx.z: 0 luma, 1 Cb+Cr) of one
// frame: warp j owns row j and hands the bottom rows of every finished macroblock to warp j+1 through a
// shared-memory line buffer (a hop of a few hundred cycles); only the first row of a CTA gets its top
// neighbours from global memory (loader warp, progress flag of the CTA above) and only the last row
// publishes its progress globally (publisher warp).
#define DB_ROWS 17
#define DB_NB 8 // line-buffer depth in macroblocks
struct DeblockRow {
    uint32_t tile[16 * 6];   // luma: 16 rows x 24 bytes (cols 0..3 = left MB's last 4 columns);
                             // chroma: 2 planes x 8 rows x 12 bytes
    uint4 lb[DB_NB][4];      // bottom rows of finished macroblocks: luma 4 rows x 16 B; chroma [plane][2 rows] x 8 B
    volatile int ready;      // macroblocks [0, ready) of lb are final (left edge of the next MB applied)
    volatile int consumed;   // this row has consumed the top neighbours of macroblocks [0, consumed)
};

// Warp-collective wait for a shared-memory counter that another warp of the CTA raises: lane 0 polls until *p >= want,
// sleeping `sleep_ns` between reads; the fence orders the warp's later reads after what the writer stored before.
__device__ __forceinline__ void spin_until_ge(volatile int *p, int want, int lane, unsigned sleep_ns)
{
    if (lane == 0)
        while (*p < want)
            __nanosleep(sleep_ns);
    __syncwarp();
    __threadfence_block();
}

// The wavefront protocol of filtering warp j, the same for both plane types: where the top neighbours of a macroblock
// come from, when its line-buffer slot may be overwritten, and the flags that report it stored.  Every member is called
// by the whole warp.
struct DeblockWave {
    DeblockRow *rows;
    DeblockMail *mail;
    uint4 (*ring)[4];
    int j, lane;
    bool has_top, top_local, below_local, publish;

    // Top neighbours of macroblock mbx from the row above's line buffer or the loader's ring; nullptr when there are
    // none, or when the line buffer's are not needed because no horizontal edge is filtered.  The ring of the CTA's
    // first row is consumed in order, so that row always waits.
    __device__ __forceinline__ uint8_t *top(int mbx, bool any_h) const
    {
        uint8_t *t = nullptr;
        if (top_local) {
            if (any_h) {
                spin_until_ge(&rows[j - 1].ready, mbx + 1, lane, 20);
                t = (uint8_t *)rows[j - 1].lb[mbx % DB_NB];
            } else
                __syncwarp();
        } else if (has_top) {
            spin_until_ge(&mail->top_ready, mbx + 1, lane, 32);
            t = (uint8_t *)ring[mbx & 1];
        } else
            __syncwarp();
        return t;
    }
    // The line-buffer slot of mbx is free once the row below has consumed macroblock mbx - DB_NB.
    __device__ __forceinline__ void wait_slot(int mbx) const
    {
        if (below_local)
            spin_until_ge(&rows[j + 1].consumed, mbx - DB_NB + 1, lane, 20);
        else
            __syncwarp();
    }
    // Macroblock mbx is stored to the frame and, for the row below, to the line buffer.
    __device__ __forceinline__ void done(int mbx) const
    {
        // the stores to the frame precede the flag: the row below stores this macroblock's bottom rows again after its
        // top edge has filtered them, and that store has to land after this one
        __threadfence_block();
        __syncwarp();
        if (lane == 0) {
            rows[j].consumed = mbx + 1;
            if (below_local)
                rows[j].ready = mbx + 1; // macroblock mbx is final: nothing in this row touches it again
            if (!top_local && has_top)
                mail->top_consumed = mbx + 1;
            if (publish)
                mail->done = mbx + 1;
        }
    }
};

__global__ void __launch_bounds__((DB_ROWS + 2) * 32) deblock_kernel(Geom g, Step s, const uint8_t *__restrict__ unf,
                                                                      uint8_t *rec, const uint8_t *__restrict__ bs,
                                                                      int *flags_y, int *flags_c, int cta_rows)
{
    if (lane_frame(s, blockIdx.y) < 0)
        return;
    __shared__ DeblockRow rows[DB_ROWS];
    __shared__ uint4 ring[2][4]; // top neighbours of the CTA's first row, staged by the loader: [slot][...]
    __shared__ DeblockMail mail;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool chroma = blockIdx.z != 0;
    const int row0 = blockIdx.x * cta_rows, nr = imin_(cta_rows, g.mbh - row0);
    const size_t fo = (size_t)blockIdx.y * g.frame_bytes;
    int *fl = (chroma ? flags_c : flags_y) + (size_t)blockIdx.y * g.mbh;
    if (threadIdx.x < DB_ROWS) {
        rows[threadIdx.x].ready = 0;
        rows[threadIdx.x].consumed = 0;
    }
    if (threadIdx.x == 0)
        mail.top_ready = mail.top_consumed = mail.done = 0;
    __syncthreads();

    if (warp == cta_rows) { // loader: top neighbours of row0 from the CTA above
        if (row0 > 0) {
            if (!chroma)
                deblock_loader(&mail, fl + row0 - 1, g.mbw, lane, [&](int slot, int mbx) {
                    if (lane < 4)
                        ring[slot][lane] = __ldcg((const uint4 *)(rec + fo + (size_t)(row0 * 16 - 4 + lane) * g.W + mbx * 16));
                });
            else
                deblock_loader(&mail, fl + row0 - 1, g.mbw, lane, [&](int slot, int mbx) {
                    if (lane < 4) {
                        int pl = lane >> 1, r = lane & 1;
                        ((uint2 *)ring[slot])[lane] =
                            __ldcg((const uint2 *)(rec + fo + (size_t)g.W * g.H + (size_t)pl * g.CW * g.CH +
                                                   (size_t)(row0 * 8 - 2 + r) * g.CW + mbx * 8));
                    }
                });
        }
        return;
    }
    if (warp == cta_rows + 1) { // publisher: progress of the CTA's last row, for the CTA below
        if (row0 + nr < g.mbh)
            deblock_publisher(&mail, fl + row0 + nr - 1, g.mbw, lane);
        return;
    }
    if (warp >= nr)
        return;

    const int j = warp, row = row0 + j;
    DeblockRow &me = rows[j];
    const bool has_top = row > 0, below_local = j + 1 < nr;
    const DeblockWave wave = {rows, &mail, ring, j, lane, has_top, j > 0, below_local, j == nr - 1 && row + 1 < g.mbh};
    const uint4 *fbs = (const uint4 *)bs + ((size_t)blockIdx.y * g.nmb + (size_t)row * g.mbw) * 2;

    if (!chroma) {
        const int sh = (lane >> 2) * 8; // byte of a strength word that belongs to this lane's 4-sample segment
        const int alpha = h264_deblock_alpha[g.qp], beta = h264_deblock_beta[g.qp];
        const int tc0_1 = h264_deblock_tc0[g.qp][0], tc0_2 = h264_deblock_tc0[g.qp][1], tc0_3 = h264_deblock_tc0[g.qp][2];
        uint8_t *tb = (uint8_t *)me.tile;
        const uint8_t *urow = unf + fo + (size_t)(row * 16 + (lane & 15)) * g.W;
        uint4 nx_px = *(const uint4 *)urow, nx_v = fbs[0], nx_h = fbs[1];
        uint32_t q0w = nx_px.x; // columns 0..3 of the macroblock about to be processed, its left edge already filtered
#ifdef DB_PROFILE
        long long pt[6] = {0, 0, 0, 0, 0, 0}, pc = clock64();
#define DB_MARK(i) { long long n_ = clock64(); pt[i] += n_ - pc; pc = n_; }
#else
#define DB_MARK(i)
#endif
        // Order inside a row (1:1 wavefront): iteration x = vertical edges 1..3 of macroblock x, its horizontal edges, then
        // vertical edge 0 of macroblock x + 1.  Every pair of edge filters with overlapping samples keeps the order of the
        // standard's raster scan (edge 0 of x + 1 touches columns 12..19 of rows of this macroblock row only: after the
        // horizontal edges of x, before edges 1..3 and the horizontal edges of x + 1), and macroblock x is FINAL when its
        // iteration ends -- the row below may start on it one iteration later, not two.
        for (int mbx = 0; mbx < g.mbw; mbx++) {
            const bool has_next = mbx + 1 < g.mbw;
            const int x0 = mbx * 16, y0 = row * 16;
            const uint4 px = nx_px, bv = nx_v, bh = nx_h;
            DB_MARK(0);
            if (has_next) { // prefetch the next macroblock
                nx_px = *(const uint4 *)(urow + x0 + 16);
                nx_v = fbs[(mbx + 1) * 2];
                nx_h = fbs[(mbx + 1) * 2 + 1];
            }
            // A phase without a single non-zero strength -- most macroblocks of a P picture with coherent motion -- is
            // passed through: the strength words are the same in every lane, so the tests are warp uniform.
            const bool any_v = (bv.y | bv.z | bv.w) != 0, any_h = (bh.x | bh.y | bh.z | bh.w) != 0;
            const bool any_vn = has_next && nx_v.x != 0;
            // ---- vertical edges 1..3, lane = row: the row's 16 pixels stay in registers ----
            if (lane < 16) {
                uint32_t *t = me.tile + lane * 6;
                uint32_t w[5] = {0u, q0w, px.y, px.z, px.w};
                if (any_v) {
                    const uint32_t bw[4] = {0u, bv.y, bv.z, bv.w};
#pragma unroll
                    for (int e = 1; e < 4; e++) {
                        int bS = (bw[e] >> sh) & 0xff;
                        if (bS) {
                            int v[8];
#pragma unroll
                            for (int i = 0; i < 4; i++)
                                v[i] = (w[e] >> (8 * i)) & 0xff, v[4 + i] = (w[e + 1] >> (8 * i)) & 0xff;
                            filter_luma8(v, bS, alpha, beta, bS == 1 ? tc0_1 : (bS == 2 ? tc0_2 : tc0_3));
                            w[e] = pack4(v);
                            w[e + 1] = pack4(v + 4);
                        }
                    }
                }
                t[1] = w[1], t[2] = w[2], t[3] = w[3], t[4] = w[4];
            }
            DB_MARK(1);
            uint8_t *top = wave.top(mbx, any_h);
            DB_MARK(2);
            // ---- horizontal edges, lane = column: the 20-sample column stays in registers ----
            if (lane < 16 && any_h) {
                uint8_t *col = tb + 4 + lane;
                int cpx[20];
#pragma unroll
                for (int i = 0; i < 4; i++)
                    cpx[i] = has_top ? top[i * 16 + lane] : 0;
#pragma unroll
                for (int i = 0; i < 16; i++)
                    cpx[4 + i] = col[i * 24];
                const uint32_t bw[4] = {bh.x, bh.y, bh.z, bh.w};
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    int bS = (bw[e] >> sh) & 0xff;
                    if (bS)
                        filter_luma8(cpx + 4 * e, bS, alpha, beta, bS == 1 ? tc0_1 : (bS == 2 ? tc0_2 : tc0_3));
                }
                if (has_top) {
#pragma unroll
                    for (int i = 1; i < 4; i++)
                        top[i * 16 + lane] = (uint8_t)cpx[i];
                }
#pragma unroll
                for (int i = 0; i < 15; i++)
                    col[i * 24] = (uint8_t)cpx[4 + i];
            }
            __syncwarp();
            // ---- vertical edge 0 of the next macroblock, lane = row: finalises columns 13..15 of this one ----
            if (lane < 16) {
                q0w = nx_px.x;
                if (any_vn) {
                    int bS = (nx_v.x >> sh) & 0xff;
                    if (bS) {
                        uint32_t *t = me.tile + lane * 6;
                        const uint32_t wp = t[4];
                        int v[8];
#pragma unroll
                        for (int i = 0; i < 4; i++)
                            v[i] = (wp >> (8 * i)) & 0xff, v[4 + i] = (q0w >> (8 * i)) & 0xff;
                        filter_luma8(v, bS, alpha, beta, bS == 1 ? tc0_1 : (bS == 2 ? tc0_2 : tc0_3));
                        t[4] = pack4(v);
                        q0w = pack4(v + 4);
                    }
                }
            }
            DB_MARK(3);
            wave.wait_slot(mbx);
            DB_MARK(4);
            if (lane < 16) {
                const uint32_t *t = me.tile + lane * 6;
                uint8_t *o = rec + fo + (size_t)(y0 + lane) * g.W + x0;
                const uint4 mine = make_uint4(t[1], t[2], t[3], t[4]);
                *(uint4 *)o = mine;
                if (below_local && lane >= 12)
                    me.lb[mbx % DB_NB][lane - 12] = mine;
            } else if (lane < 19 && has_top && any_h) {
                int r = lane - 15; // top rows 1..3 were modified
                *(uint4 *)(rec + fo + (size_t)(y0 - 4 + r) * g.W + x0) = ((const uint4 *)top)[r];
            }
            wave.done(mbx);
            DB_MARK(5);
        }
#ifdef DB_PROFILE
        if (lane == 0 && blockIdx.y == 0 && (row == 20 || row == 24))
            printf("deblock luma row %d: cycles per MB: prefetch %lld  V-edges %lld  flag+wait-top %lld  H-edges %lld  wait-slot %lld  store+flags %lld\n",
                   row, pt[0] / g.mbw, pt[1] / g.mbw, pt[2] / g.mbw, pt[3] / g.mbw, pt[4] / g.mbw, pt[5] / g.mbw);
#endif
#undef DB_MARK
    } else {
        const int alpha = h264_deblock_alpha[g.qpc], beta = h264_deblock_beta[g.qpc];
        const int tc0_1 = h264_deblock_tc0[g.qpc][0], tc0_2 = h264_deblock_tc0[g.qpc][1], tc0_3 = h264_deblock_tc0[g.qpc][2];
        const int pl = (lane >> 3) & 1, r8 = lane & 7;
        const size_t po = fo + (size_t)g.W * g.H + (size_t)pl * g.CW * g.CH;
        uint32_t *tw = me.tile + pl * 24;
        uint8_t *tb = (uint8_t *)tw;
        const int shc = (r8 >> 1) * 8; // chroma row / column k <-> luma segment k >> 1
        const uint8_t *urow = unf + po + (size_t)(row * 8 + r8) * g.CW;
        uint2 nx_px = *(const uint2 *)urow;
        uint4 nx_v = fbs[0], nx_h = fbs[1];
        uint32_t q0w = nx_px.x; // columns 0..3 of the macroblock about to be processed, its left edge already filtered
        // same order as the luma path: vertical edge at x = 4, horizontal edges, vertical edge at x = 0 of the next macroblock
        for (int mbx = 0; mbx < g.mbw; mbx++) {
            const bool has_next = mbx + 1 < g.mbw;
            const int x0 = mbx * 8, y0 = row * 8;
            const uint2 px = nx_px;
            const uint4 bv = nx_v, bh = nx_h;
            if (has_next) {
                nx_px = *(const uint2 *)(urow + x0 + 8);
                nx_v = fbs[(mbx + 1) * 2];
                nx_h = fbs[(mbx + 1) * 2 + 1];
            }
            const bool any_v = bv.z != 0, any_h = (bh.x | bh.z) != 0; // warp uniform, as in the luma path
            const bool any_vn = has_next && nx_v.x != 0;
            if (lane < 16) { // vertical edge at chroma x = 4 (luma edge 2): lane = (plane, row)
                uint32_t *t = tw + r8 * 3;
                uint32_t w1 = q0w, w2 = px.y;
                if (any_v) {
                    int bS = (bv.z >> shc) & 0xff;
                    if (bS) {
                        int v[4] = {(int)((w1 >> 16) & 0xff), (int)(w1 >> 24), (int)(w2 & 0xff), (int)((w2 >> 8) & 0xff)};
                        filter_chroma4(v, bS, alpha, beta, bS == 1 ? tc0_1 : (bS == 2 ? tc0_2 : tc0_3));
                        w1 = (w1 & 0x00ffffffu) | ((uint32_t)v[1] << 24);
                        w2 = (w2 & 0xffffff00u) | (uint32_t)v[2];
                    }
                }
                t[1] = w1, t[2] = w2;
            }
            uint8_t *topb = wave.top(mbx, any_h); // [plane][2 rows][8 bytes]
            uint8_t *top = topb + pl * 16;
            if (lane < 16 && any_h) { // horizontal edges at chroma y = 0, 4: lane = (plane, column)
                uint8_t *col = tb + 4 + r8;
                int cpx[8];
                cpx[0] = has_top ? top[r8] : 0;
                cpx[1] = has_top ? top[8 + r8] : 0;
#pragma unroll
                for (int i = 0; i < 6; i++)
                    cpx[2 + i] = col[i * 12];
                const uint32_t bw[2] = {bh.x, bh.z};
#pragma unroll
                for (int ce = 0; ce < 2; ce++) {
                    int bS = (bw[ce] >> shc) & 0xff;
                    if (bS)
                        filter_chroma4(cpx + 4 * ce, bS, alpha, beta, bS == 1 ? tc0_1 : (bS == 2 ? tc0_2 : tc0_3));
                }
                if (has_top)
                    top[8 + r8] = (uint8_t)cpx[1];
                col[0 * 12] = (uint8_t)cpx[2];
                col[3 * 12] = (uint8_t)cpx[5];
                col[4 * 12] = (uint8_t)cpx[6];
            }
            __syncwarp();
            if (lane < 16) { // vertical edge at x = 0 of the next macroblock: finalises column 7 of this one
                q0w = nx_px.x;
                if (any_vn) {
                    int bS = (nx_v.x >> shc) & 0xff;
                    if (bS) {
                        uint32_t *t = tw + r8 * 3;
                        const uint32_t wp = t[2];
                        int v[4] = {(int)((wp >> 16) & 0xff), (int)(wp >> 24), (int)(q0w & 0xff), (int)((q0w >> 8) & 0xff)};
                        filter_chroma4(v, bS, alpha, beta, bS == 1 ? tc0_1 : (bS == 2 ? tc0_2 : tc0_3));
                        t[2] = (wp & 0x00ffffffu) | ((uint32_t)v[1] << 24);
                        q0w = (q0w & 0xffffff00u) | (uint32_t)v[2];
                    }
                }
            }
            wave.wait_slot(mbx);
            if (lane < 16) {
                uint8_t *o = rec + po + (size_t)(y0 + r8) * g.CW + x0;
                const uint2 mine = make_uint2(tw[r8 * 3 + 1], tw[r8 * 3 + 2]);
                *(uint2 *)o = mine;
                if (below_local && r8 >= 6)
                    ((uint2 *)me.lb[mbx % DB_NB])[pl * 2 + (r8 - 6)] = mine;
            } else if (lane < 18 && has_top && any_h) {
                int p2 = lane - 16;
                *(uint2 *)(rec + fo + (size_t)g.W * g.H + (size_t)p2 * g.CW * g.CH + (size_t)(y0 - 1) * g.CW + x0) =
                    ((const uint2 *)topb)[p2 * 2 + 1];
            }
            wave.done(mbx);
        }
    }
}

// ================================================================================================
// K9 statistics: sum of squared luma error per frame (exact integer), for Y-PSNR.
// ================================================================================================
__global__ void sse_kernel(Geom g, Step s, const uint8_t *__restrict__ src, const uint8_t *__restrict__ rec,
                           unsigned long long *__restrict__ sse)
{
    int f = lane_frame(s, blockIdx.y);
    if (f < 0)
        return;
    const size_t fo = (size_t)blockIdx.y * g.frame_bytes, n4 = (size_t)g.W * g.H / 4;
    unsigned acc = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        uint32_t a = ((const uint32_t *)(src + fo))[i], b = ((const uint32_t *)(rec + fo))[i];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            int d = (int)((a >> (8 * k)) & 0xff) - (int)((b >> (8 * k)) & 0xff);
            acc += (unsigned)(d * d);
        }
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1)
        acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0)
        atomicAdd(sse + f, (unsigned long long)acc);
}

// ================================================================================================
// K6 / K7 entropy coding, pass structure: sizes per macroblock -> exclusive prefix sum per frame ->
// scatter.  CAVLC scatters bits; CABAC scatters bins and a serial arithmetic coder (one per frame,
// many frames at once) turns them into bytes.
// ================================================================================================
// "Unit" = one slice NAL: unit index u = frame * nslices + slice (nslices = 1 in the reference's layout).
struct EntropyBufs {
    uint32_t *mb_size;       // [L][nitems + 1] bits (CAVLC) or bins (CABAC) per entropy item (slice_item)
    uint32_t *mb_off;        // [L][nitems + 1] exclusive prefix over the picture; [nitems] = total
    const unsigned long long *hdr_bits; // [U] slice header bits (host written, cedar.c:984-1030)
    const int *hdr_nbits;     // [U]
    uint8_t *rbsp;           // [U][rbsp_cap]
    unsigned rbsp_cap;
    uint32_t *rbsp_len;      // [U] bytes of RBSP (header + slice data + trailing)
    uint16_t *bins;          // CABAC bin pool
    unsigned long long bins_cap;
    unsigned long long *bins_cursor; // pool bump pointer
    unsigned long long *bins_off;    // [U]
    uint32_t *bins_len;      // [U]
    uint32_t *limbs;         // [coder CTAs of one launch][limb_cap] code-word limbs of the CABAC coder (16 stream bits per
                             // 32-bit word): scratch of the launch, one region per side stream (set by the host)
    unsigned long long limb_cap;
    int *error;              // sticky overflow flag
    const uint8_t *i4;       // [L][nmb][16] Intra4x4 prediction modes of the step being coded (intra4x4 extension)
};

__device__ __forceinline__ FrameSyntax lane_syntax(const Geom &g, int lane, const MbInfo *mbi, const uint8_t *nnz,
                                                   const int16_t *coef, const uint8_t *i4 = nullptr)
{
    FrameSyntax fs;
    fs.mbi = mbi + (size_t)lane * g.nmb;
    fs.nnz = nnz + (size_t)lane * g.nmb * NNZ_STRIDE;
    fs.coef = coef + (size_t)lane * g.nmb * COEF_STRIDE;
    fs.mbw = g.mbw;
    fs.mbh = g.mbh;
    fs.srows = g.srows;
    fs.i4 = i4 ? i4 + (size_t)lane * g.nmb * 16 : nullptr;
    return fs;
}

__global__ void entropy_size_kernel(Geom g, Step s, int frame_i, const MbInfo *__restrict__ mbi,
                                    const uint8_t *__restrict__ nnz, const int16_t *__restrict__ coef, EntropyBufs eb)
{
    if (lane_frame(s, blockIdx.y) < 0)
        return;
    const int nitems = g.nmb + g.nslices;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nitems)
        return;
    FrameSyntax fs = lane_syntax(g, blockIdx.y, mbi, nnz, coef, eb.i4);
    const SliceItem it = slice_item(fs, i);
    unsigned n;
    if (g.cabac) {
        BinCount c;
        if (!it.is_end)
            cabac_mb(c, fs, it.mb, frame_i);
        n = c.n;
    } else {
        BitCount c;
        if (it.is_end)
            cavlc_end(c, frame_i ? 0 : skip_run_before(fs, it.mb, it.first_mb));
        else if (fs.mbi[it.mb].type != MB_PSKIP)
            cavlc_mb(c, fs, it.mb, frame_i, frame_i ? 0 : skip_run_before(fs, it.mb, it.first_mb));
        n = c.n;
    }
    eb.mb_size[(size_t)blockIdx.y * (nitems + 1) + i] = n;
}

// Exclusive scan of in[0, n) into out[0, n) by one 1024-thread CTA, starting at `carry`, in chunks of 1024: a warp scan,
// a scan of the warp sums, then the carry into the next chunk.  Each thread reads its element before it writes it, so
// in == out is allowed.  Returns carry + the sum of in[0, n) to every thread.
template <class In, class Acc>
__device__ __forceinline__ Acc block_exclusive_scan(const In *in, Acc *out, unsigned n, Acc carry)
{
    __shared__ Acc warp_sum[32];
    __shared__ Acc carry_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0)
        carry_s = carry;
    __syncthreads();
    for (unsigned start = 0; start < n; start += 1024) {
        const unsigned i = start + tid;
        Acc v = i < n ? (Acc)in[i] : 0, x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            Acc y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o)
                x += y;
        }
        if (lane == 31)
            warp_sum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            Acc ws = warp_sum[lane], z = ws;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                Acc y = __shfl_up_sync(0xffffffffu, z, o);
                if (lane >= o)
                    z += y;
            }
            warp_sum[lane] = z - ws; // exclusive
        }
        __syncthreads();
        Acc incl = carry_s + warp_sum[warp] + x;
        if (i < n)
            out[i] = incl - v;
        __syncthreads();
        if (tid == 1023)
            carry_s = incl;
        __syncthreads();
    }
    return carry_s;
}

// Exclusive prefix sum of the item sizes of a picture (one 1024-thread CTA per lane) + per-slice totals.
__global__ void __launch_bounds__(1024) entropy_scan_kernel(Geom g, Step s, EntropyBufs eb)
{
    int f = lane_frame(s, blockIdx.y);
    if (f < 0)
        return;
    __shared__ unsigned long long pool_off;
    const int n = g.nmb + g.nslices, tid = threadIdx.x;
    uint32_t *out = eb.mb_off + (size_t)blockIdx.y * (n + 1);
    const uint32_t total = block_exclusive_scan(eb.mb_size + (size_t)blockIdx.y * (n + 1), out, n, 0u);
    if (tid == 0) {
        out[n] = total;
        if (g.cabac) { // one pool allocation per picture; its slices lie back to back
            unsigned long long off = atomicAdd(eb.bins_cursor, (unsigned long long)((total + 7u) & ~7u));
            if (off + total > eb.bins_cap) {
                atomicExch(eb.error, 1);
                off = ~0ull;
            }
            pool_off = off;
        }
    }
    __syncthreads();
    const int per = g.srows * g.mbw + 1;
    for (int k = tid; k < g.nslices; k += 1024) {
        const size_t u = (size_t)f * g.nslices + k;
        const uint32_t start = out[k * per], end = out[imin_((k + 1) * per, n)];
        if (g.cabac) {
            eb.bins_off[u] = pool_off == ~0ull ? 0 : pool_off + start;
            eb.bins_len[u] = pool_off == ~0ull ? 0 : end - start;
        } else {
            uint32_t bytes = ((uint32_t)eb.hdr_nbits[u] + (end - start) + 7) >> 3;
            if (bytes + 8 > eb.rbsp_cap) {
                atomicExch(eb.error, 2);
                bytes = 0;
            }
            eb.rbsp_len[u] = bytes;
        }
    }
}

__global__ void entropy_write_kernel(Geom g, Step s, int frame_i, const MbInfo *__restrict__ mbi,
                                     const uint8_t *__restrict__ nnz, const int16_t *__restrict__ coef, EntropyBufs eb)
{
    int f = lane_frame(s, blockIdx.y);
    if (f < 0)
        return;
    const int nitems = g.nmb + g.nslices;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nitems)
        return;
    FrameSyntax fs = lane_syntax(g, blockIdx.y, mbi, nnz, coef, eb.i4);
    const SliceItem it = slice_item(fs, i);
    const uint32_t *offs = eb.mb_off + (size_t)blockIdx.y * (nitems + 1);
    const uint32_t off = offs[i] - offs[it.slice * slice_items_per(fs)]; // relative to the slice's first item
    const size_t u = (size_t)f * g.nslices + it.slice;
    if (g.cabac) {
        if (it.is_end || eb.bins_len[u] == 0)
            return;
        BinWrite w(eb.bins + eb.bins_off[u] + off);
        cabac_mb(w, fs, it.mb, frame_i);
    } else {
        if (eb.rbsp_len[u] == 0)
            return;
        uint32_t *buf = (uint32_t *)(eb.rbsp + u * eb.rbsp_cap);
        const int hn = eb.hdr_nbits[u];
        if (it.is_first) { // slice header bits (up to 46 with first_mb_in_slice != 0)
            BitScatter h(buf, 0);
            const unsigned long long hb = eb.hdr_bits[u];
            if (hn > 32)
                h.put((uint32_t)(hb >> 32), hn - 32);
            h.put((uint32_t)hb, hn > 32 ? 32 : hn);
            h.flush();
        }
        if (!it.is_end && fs.mbi[it.mb].type == MB_PSKIP)
            return;
        BitScatter w(buf, (unsigned long long)hn + off);
        if (it.is_end)
            cavlc_end(w, frame_i ? 0 : skip_run_before(fs, it.mb, it.first_mb));
        else
            cavlc_mb(w, fs, it.mb, frame_i, frame_i ? 0 : skip_run_before(fs, it.mb, it.first_mb));
        w.flush();
    }
}

// K7 CABAC arithmetic coding, one slice per CTA (one slice per picture in the reference's layout,
// cedar.c:992-993), in two kernels; entropy.cuh derives the parallel formulation.
//
// cabac_resolve_kernel: context-state resolution.  The state a regular bin is coded in depends only on the
// earlier bins of the same context, so the work is a set of independent serial chains, one per context (460 of
// them; the hottest holds about 6 % of a slice's bins).  One CTA per slice; every context is OWNED by one thread
// that keeps its state in a register for the whole slice.  Per tile of RES_TILE bins:
//   A. stable counting sort by context, first half: every warp ranks the bins of its contiguous 256-bin chunk, 32 at a
//      time -- nine ballots give each lane the lanes holding the same context, the lowest of them bumps the warp's own
//      counter of that context (no atomics: a counter row belongs to one warp, one leader per context per step);
//   B. the owner of a context turns its column of the counters into offsets (exclusive prefix over the warps) and the
//      block scans the per-context totals, rounded up to 32, into the start of every context's segment;
//   C. every bin's VALUE goes to its place in the sorted order (a bit array; one shared atomic OR per 1-bin);
//   D. the owner walks its segment FOUR bins per dependent table look-up: the 128-state machine composed four times
//      (2048 entries of 16 bytes: the four records -- cabac_meta: isLPS + pStateIdx -- and the state after them), the
//      records stored in sorted order with one 8-byte store.  Chain per four bins: OR, shift, LDS.128;
//   E. every bin fetches its record from its place in the sorted order.
// The only serial part is D along one context; its length per tile is the hottest context's bin count / 4.
// Bounds-check build (-DCEDAR_B200_BOUNDS; compute-sanitizer is closed on the pool): every computed shared-memory index of
// the resolver is asserted before use; a violation prints where and traps.  tools/san_case.py and the 1080p parity tests
// run clean under it (profiles/r02_bounds_build.txt).
#ifdef CEDAR_B200_BOUNDS
#define RES_ASSERT(cond, what, val)                                                                                  \
    do {                                                                                                             \
        if (!(cond)) {                                                                                               \
            printf("cabac_resolve_kernel: %s out of bounds: %u (block %d thread %d)\n", what, (unsigned)(val), blockIdx.x, \
                   threadIdx.x);                                                                                     \
            __trap();                                                                                                \
        }                                                                                                            \
    } while (0)
#else
#define RES_ASSERT(cond, what, val)
#endif
__device__ __forceinline__ uint4 lds_u128(uint32_t addr)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_u64(uint32_t addr, uint32_t a, uint32_t b)
{
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}
#define RES_WARPS 16
#define RES_THREADS (RES_WARPS * 32)
#define RES_TILE 4096
#define RES_GROUPS (RES_TILE / 32)
#define RES_GPW (RES_GROUPS / RES_WARPS)   // 32-bin groups per warp and tile
#define RES_NCTX 464                       // 460 contexts, padded
#define RES_SORTED (RES_TILE + 31 * RES_NCTX + 32) // sorted order with every segment padded to a multiple of 32
#define RES_TAB_BYTES (2048 * 16)
#define RES_SMEM_BYTES (RES_TAB_BYTES + (RES_TILE + 8) * 2 + RES_SORTED * 2 + (RES_SORTED / 32 + 2) * 4)
__global__ void __launch_bounds__(RES_THREADS) cabac_resolve_kernel(Geom g, Step s, int gop_len, int gop_pos0,
                                                                    EntropyBufs eb, unsigned long long *ctx_hist)
{
    extern __shared__ __align__(16) uint8_t res_dyn[];            // RES_SMEM_BYTES
    uint4 *const step4 = (uint4 *)res_dyn;                        // [state << 4 | four bin values]
    uint16_t *const tile = (uint16_t *)(res_dyn + RES_TAB_BYTES); // [RES_TILE + 8] bins in, records out
    uint16_t *const recq = tile + RES_TILE + 8;                   // [RES_SORTED] records in sorted order
    uint32_t *const bitq = (uint32_t *)(recq + RES_SORTED);       // [RES_SORTED / 32 + 2] bin values in sorted order
    __shared__ uint16_t wcnt[RES_WARPS][RES_NCTX]; // [w][slot(c)]: bins of context c in warp w's chunk -> exclusive prefix over w
    __shared__ uint16_t cstart[RES_NCTX];
    __shared__ uint16_t wsum[RES_WARPS];
    const int f = lane_frame(s, blockIdx.x / g.nslices); // one CTA per slice
    if (f < 0)
        return;
    const size_t u = (size_t)f * g.nslices + blockIdx.x % g.nslices;
    const uint32_t nb = eb.bins_len[u];
    if (nb == 0)
        return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t lt = (1u << lane) - 1;
    const int frame_i = ((gop_pos0 + f) % gop_len) == 0;
    uint16_t *gb = eb.bins + eb.bins_off[u];
    // 16-byte vector loads / stores: tile k starts at the aligned address at or below gb + k * RES_TILE
    const uint32_t mis = (uint32_t)(((uintptr_t)gb >> 1) & 7); // elements between that address and the first bin
    // step4[(pStateIdx << 1 | valMPS) << 4 | b0 | b1 << 1 | b2 << 2 | b3 << 3]:
    //   .x = record of bin 0 | record of bin 1 << 16, .y = records of bins 2 and 3, .z = state after the four bins << 4.
    // The record of a bin coded in state S is (pStateIdx << 3 | valMPS) ^ value: bit 0 = isLPS, bits 3.. = pStateIdx.
    for (int idx = tid; idx < 2048; idx += RES_THREADS) {
        uint32_t st7 = idx >> 4, rec[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t ps = st7 >> 1, mps = st7 & 1, bit = (idx >> j) & 1;
            rec[j] = ((ps << 3) | mps) ^ bit;
            if (bit == mps)
                st7 = ((ps < 62 ? ps + 1 : ps) << 1) | mps; // h264_next_state_mps
            else
                st7 = (h264_next_state_lps[ps] << 1) | (ps == 0 ? mps ^ 1 : mps);
        }
        step4[idx] = make_uint4(rec[0] | (rec[1] << 16), rec[2] | (rec[3] << 16), st7 << 4, 0);
    }
    // Thread (warp, lane < 29) owns context lane * 16 + warp: neighbouring contexts -- the hot ones come in runs
    // (significance flags 105.., levels 227..) -- sit in different warps.  Counters and segment starts are stored at
    // slot(c) = (c & 15) * 29 + (c >> 4) = warp * 29 + lane of the owner, which pass B reads conflict free.
    const int myc = lane < 29 ? lane * 16 + warp : 511, myslot = warp * 29 + lane;
    uint32_t X = myc < 460 ? cabac_init_state(myc, frame_i, g.qp) << 4 : 0; // (pStateIdx << 1 | valMPS) << 4
    // shared-window addresses for the walk of pass D, made opaque so that they stay in registers (otherwise they are
    // rebuilt from SR_CgaCtaId, a 20-cycle special-register read, inside the loop)
    uint32_t tab_addr = (uint32_t)__cvta_generic_to_shared(step4), recq_addr = (uint32_t)__cvta_generic_to_shared(recq);
    uint32_t bitq_addr = (uint32_t)__cvta_generic_to_shared(bitq);
    asm volatile("mov.u32 %0, %0;" : "+r"(tab_addr));
    asm volatile("mov.u32 %0, %0;" : "+r"(recq_addr));
    asm volatile("mov.u32 %0, %0;" : "+r"(bitq_addr));
#ifdef RES_PROFILE
    __shared__ unsigned long long prof_acc[8], prof_dmax, prof_dsum, prof_cnt;
    long long prof_t = clock64();
    if (tid < 8)
        prof_acc[tid] = 0;
    if (tid == 0)
        prof_dmax = 0, prof_dsum = 0, prof_cnt = 0;
#define RES_PROF_MARK(i)                                                                                       \
    {                                                                                                          \
        const long long now_ = clock64();                                                                      \
        if (tid == 0) {                                                                                        \
            prof_acc[i] += (unsigned long long)(now_ - prof_t);                                                \
            if ((i) == 4) {                                                                                    \
                prof_dsum += (prof_dmax >> 8) & 0xfff;                                                         \
                prof_cnt++;                                                                                    \
                prof_dmax = 0;                                                                                 \
            }                                                                                                  \
        }                                                                                                      \
        prof_t = now_;                                                                                         \
    }
#else
#define RES_PROF_MARK(i)
#endif
    for (uint32_t base = 0; base < nb; base += RES_TILE) {
        const uint32_t n = nb - base < RES_TILE ? nb - base : RES_TILE;
        const uint16_t *src = gb + base - mis; // 16-byte aligned
        const uint32_t nv = (mis + n + 7) >> 3;
        __syncthreads(); // table ready / previous tile's records stored
        for (uint32_t v = tid; v < nv; v += RES_THREADS) {
            // the first and the last vector may reach into a neighbouring slice's bins (same pool): read-only here
            ((uint4 *)tile)[v] = ((const uint4 *)src)[v];
        }
        for (int i = tid; i < RES_WARPS * RES_NCTX / 2; i += RES_THREADS)
            ((uint32_t *)wcnt)[i] = 0;
        for (int i = tid; i < RES_SORTED / 32 + 2; i += RES_THREADS)
            bitq[i] = 0;
        __syncthreads();
        RES_PROF_MARK(0);
        // ---- A. rank inside the warp's chunk ----
        uint32_t ent[RES_GPW]; // slot | value << 9 | rank in chunk << 10; 0xffffffff = not a regular bin
#pragma unroll
        for (int gi = 0; gi < RES_GPW; gi++) {
            const uint32_t i = (warp * RES_GPW + gi) * 32 + lane;
            const bool live = i < n;
            const uint32_t b = live ? tile[mis + i] : (uint32_t)BIN_BYPASS;
            const bool reg = !(b & (BIN_BYPASS | BIN_TERM));
            const uint32_t c = b & 0x3ff;
            if (live && !reg)
                tile[mis + i] = cabac_meta((uint16_t)b, 0);
            // lanes holding the same context: nine ballots (match.any takes hundreds of cycles per call here)
            uint32_t peers = __ballot_sync(0xffffffffu, reg);
#pragma unroll
            for (int bit = 0; bit < 9; bit++) {
                const int sh = (int)(c << (31 - bit)); // bit `bit` of c in the sign: one shift feeds the vote and the mask
                const uint32_t bb = __ballot_sync(0xffffffffu, sh < 0);
                peers &= ~(bb ^ (uint32_t)(sh >> 31));
            }
            if (!reg)
                peers = 1u << lane;
            uint32_t cbase = 0;
            const uint32_t slot = (c & 15) * 29 + (c >> 4);
            RES_ASSERT(!reg || (c < 460 && slot < RES_NCTX), "context / slot", c);
            if (reg && !(peers & lt)) { // lowest lane holding context c: this step's only writer of wcnt[warp][slot]
                cbase = wcnt[warp][slot];
                wcnt[warp][slot] = (uint16_t)(cbase + __popc(peers));
            }
            cbase = __shfl_sync(0xffffffffu, cbase, __ffs(peers) - 1);
            ent[gi] = reg ? (slot | (((b >> 15) & 1) << 9) | ((cbase + __popc(peers & lt)) << 10)) : 0xffffffffu;
            __syncwarp();
        }
        __syncthreads();
        RES_PROF_MARK(1);
        // ---- B. offsets: over the warps per context, over the contexts (segments padded to multiples of four) ----
        uint32_t total = 0;
        if (lane < 29) {
#pragma unroll
            for (int w = 0; w < RES_WARPS; w++) {
                const uint32_t v = wcnt[w][myslot];
                wcnt[w][myslot] = (uint16_t)total;
                total += v;
            }
        }
        const uint32_t padded = (total + 31) & ~31u; // a segment starts on a word of the bit array
        uint32_t incl = padded;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o)
                incl += y;
        }
        if (lane == 31)
            wsum[warp] = (uint16_t)incl;
        __syncthreads();
        uint32_t qs = incl - padded; // start of this thread's context's segment, a multiple of 32
        for (int w = 0; w < warp; w++)
            qs += wsum[w];
        if (lane < 29)
            cstart[myslot] = (uint16_t)qs;
        __syncthreads();
        RES_PROF_MARK(2);
        // ---- C. the bin values in sorted order; ent[] becomes the bin's position there ----
#pragma unroll
        for (int gi = 0; gi < RES_GPW; gi++) {
            const uint32_t e = ent[gi];
            if (e != 0xffffffffu) {
                const uint32_t c = e & 0x1ff, pos = cstart[c] + wcnt[warp][c] + (e >> 10);
                RES_ASSERT(c < RES_NCTX && pos < RES_SORTED, "sorted position", pos);
                if (e & 0x200)
                    atomicOr(&bitq[pos >> 5], 1u << (pos & 31));
                ent[gi] = pos;
            }
        }
        __syncthreads();
        RES_PROF_MARK(3);
        if (ctx_hist && total) // measurement only (profiling on): bins per context, for the serial-chain bound
            atomicAdd(&ctx_hist[myc], (unsigned long long)total);
        // ---- D. the owner walks its segment, four bins per look-up ----
        {
#ifdef RES_PROFILE
            const long long d0 = clock64();
#endif
            // A segment starts on a word of the bit array: one word = the values of eight groups of four bins.  The chain
            // per group is OR, shift, LDS.128; everything else (the word of the next eight groups, the nibble, the
            // store of the four records) is off the chain, and the eight groups of a word are unrolled.
            uint32_t k = qs;
            const uint32_t kfull = qs + (total & ~3u);
            RES_ASSERT((qs & 31) == 0 && qs + ((total + 31) & ~31u) <= RES_SORTED && (X >> 4) < 128, "segment / state", qs);
            uint32_t w = lds_u32(bitq_addr + (k >> 3));
            while (k < kfull) {
                const uint32_t wn = lds_u32(bitq_addr + (k >> 3) + 4); // next word (the array is padded)
                const uint32_t ng = (kfull - k) >> 2;                   // full groups left in this segment
#pragma unroll
                for (int j = 0; j < 8; j++)
                    if ((uint32_t)j < ng) {
                        RES_ASSERT((X | 15) < 2048 && k + 4 * j + 3 < RES_SORTED, "table / record index", X);
                        const uint4 t = lds_u128(tab_addr + ((X | ((w >> (4 * j)) & 15)) << 4));
                        sts_u64(recq_addr + 2 * k + 8 * j, t.x, t.y);
                        X = t.z;
                    }
                w = wn;
                k += 32;
            }
            if (total & 3) { // one to three bins left (padding values are 0): the state after `left` bins is the state
                const uint32_t left = total & 3; // the next, padding, bin would be coded in, i.e. its record
                const uint32_t nib = (lds_u32(bitq_addr + ((kfull >> 5) << 2)) >> (kfull & 31)) & 15;
                const uint4 t = lds_u128(tab_addr + ((X | nib) << 4));
                sts_u64(recq_addr + 2 * kfull, t.x, t.y);
                const uint32_t sr = (left == 1 ? t.x >> 16 : (left == 2 ? t.y : t.y >> 16)) & 0xffff;
                X = ((sr >> 3) << 5) | ((sr & 1) << 4);
            }
#ifdef RES_PROFILE
            atomicMax(&prof_dmax, ((unsigned long long)(clock64() - d0) << 20) | (total << 8) | (unsigned)warp);
#endif
        }
        __syncthreads();
        RES_PROF_MARK(4);
        // ---- E. every regular bin fetches its record ----
#pragma unroll
        for (int gi = 0; gi < RES_GPW; gi++)
            if (ent[gi] != 0xffffffffu) {
                RES_ASSERT(ent[gi] < RES_SORTED && mis + (warp * RES_GPW + gi) * 32 + lane < RES_TILE + 8, "record fetch", ent[gi]);
                tile[mis + (warp * RES_GPW + gi) * 32 + lane] = recq[ent[gi]];
            }
        __syncthreads();
        // records back in place of the bins; the partial vectors at both ends are written element-wise
        uint16_t *dst = gb + base - mis;
        for (uint32_t v = tid; v < nv; v += RES_THREADS) {
            const uint32_t e0 = v * 8;
            if (e0 >= mis && e0 + 8 <= mis + n)
                ((uint4 *)dst)[v] = ((const uint4 *)tile)[v];
            else
                for (uint32_t e = e0 > mis ? e0 : mis; e < e0 + 8 && e < mis + n; e++)
                    dst[e] = tile[e];
        }
        RES_PROF_MARK(5);
    }
#ifdef RES_PROFILE
    if (tid == 0 && blockIdx.x == 0)
        printf("resolve profile (CTA 0, %u bins, %llu tiles): load %llu  A %llu  B %llu  C %llu  D %llu  E+store %llu cycles per tile; "
               "slowest chain avg %llu bins\n", nb, prof_cnt, prof_acc[0] / prof_cnt, prof_acc[1] / prof_cnt, prof_acc[2] / prof_cnt,
               prof_acc[3] / prof_cnt, prof_acc[4] / prof_cnt, prof_acc[5] / prof_cnt, prof_dsum / prof_cnt);
#endif
#undef RES_PROF_MARK
}

// cabac_code_kernel: the arithmetic coder proper, all bins of the slice in parallel (entropy.cuh, "parallel
// formulation").  Per tile of CP_THREADS chunks x CP_K bins: stage the records in shared memory; find the
// chunk starts (right after the first LPS bin of each CP_K-bin stretch); walk every chunk for the four
// hypotheses; scan the chunk maps; walk again with the true start range, every thread collecting its values in
// two limb registers and adding them to the slice's limb array when it moves on (few global reductions);
// finally one carry-lookahead pass over the limbs writes the bytes.  CP_K = 62 bins = 31 words: the strided
// walks are bank-conflict free.  16 warps per CTA: both walks are latency bound per thread.
#define CP_THREADS 512
#define CP_WARPS (CP_THREADS / 32)
#define CP_K 62
#define CP_TB (CP_THREADS * CP_K)
#define CP_SMEM_BYTES ((CP_TB + CP_K + 16) * 2)
__device__ __forceinline__ ChunkMap shfl_up_map(const ChunkMap &m, int off)
{
    ChunkMap o;
    o.qmap = __shfl_up_sync(0xffffffffu, m.qmap, off);
#pragma unroll
    for (int h = 0; h < 4; h++)
        o.s[h] = __shfl_up_sync(0xffffffffu, m.s[h], off);
    return o;
}

__global__ void __launch_bounds__(CP_THREADS) cabac_code_kernel(Geom g, Step s, EntropyBufs eb)
{
    extern __shared__ __align__(16) uint16_t meta_raw[]; // [CP_TB + CP_K + 16]
    __shared__ uint2 rtab[64];
    __shared__ int start_s[CP_THREADS + 1];
    __shared__ uint32_t wmap_s[CP_WARPS][5];
    __shared__ uint32_t carry_q, carry_P, wg_s[CP_WARPS], wp_s[CP_WARPS], cin_s;
    const int f = lane_frame(s, blockIdx.x / g.nslices);
    if (f < 0)
        return;
    const size_t u = (size_t)f * g.nslices + blockIdx.x % g.nslices;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nb = (int)eb.bins_len[u];
    if (nb == 0) {
        if (tid == 0)
            eb.rbsp_len[u] = 0;
        return;
    }
    const uint16_t *mg = eb.bins + eb.bins_off[u];
    const int mis = (int)(((uintptr_t)mg >> 1) & 7);
    const uint16_t *meta_s = meta_raw + mis; // meta_s[i - lo] = record of bin i
    uint32_t *limbs = eb.limbs + (size_t)blockIdx.x * eb.limb_cap;
    uint8_t *out = eb.rbsp + u * eb.rbsp_cap;
    const int hn = eb.hdr_nbits[u], hb = (hn + 7) >> 3;
    if (tid == 64) { // header bits, then cabac_alignment_one_bit up to the byte boundary
        unsigned long long h = (eb.hdr_bits[u] << (hb * 8 - hn)) | ((1ull << (hb * 8 - hn)) - 1);
        for (int i = 0; i < hb; i++)
            out[i] = (uint8_t)(h >> (8 * (hb - 1 - i)));
    }
    if (tid < 64) {
        uint32_t w = 0, sh = 0;
        for (int q = 0; q < 4; q++) {
            uint32_t lps = h264_range_lps[tid][q];
            w |= lps << (8 * q);
            sh |= (uint32_t)(8 - ilog2_(lps)) << (3 * q);
        }
        rtab[tid] = make_uint2(w, sh);
    }
    if (tid == 0)
        carry_q = 0, carry_P = 0;
    int prev_hi = -1; // limbs [0, prev_hi] are initialised (uniform over the CTA)
    bool overflow = false;
    const int ntiles = (nb + CP_TB - 1) / CP_TB;
    for (int tile = 0; tile < ntiles; tile++) {
        const int lo = tile * CP_TB, n_load = imin_(CP_TB + CP_K, nb - lo);
        __syncthreads();
        {
            const uint4 *src = (const uint4 *)(mg + lo - mis); // 16-byte aligned; may start / end in a neighbour's bins
            const int nv = (mis + n_load + 7) >> 3;
            for (int v = tid; v < nv; v += CP_THREADS)
                ((uint4 *)meta_raw)[v] = src[v];
        }
        __syncthreads();
        auto M = [&](int i) -> uint32_t { return i - lo < n_load ? meta_s[i - lo] : mg[i]; };
        // ---- chunk starts; entry CP_THREADS = first chunk start of the tiles that follow (or nb) ----
        for (int c = tid; c <= CP_THREADS; c += CP_THREADS) {
            const int lo_c = lo + c * CP_K;
            int st = -1;
            if (tile == 0 && c == 0)
                st = 0;
            else if (lo_c < nb) {
                const int hi_c = imin_(nb, lo_c + CP_K);
                for (int i = lo_c; i < hi_c; i++)
                    if (cabac_meta_is_lps(meta_s[i - lo])) {
                        st = i + 1 < nb ? i + 1 : -1;
                        break;
                    }
                if (c == CP_THREADS && st < 0) // rare: no LPS bin in the look-ahead stretch
                    for (int i = hi_c; i < nb; i++)
                        if (cabac_meta_is_lps(mg[i])) {
                            st = i + 1;
                            break;
                        }
            }
            if (c == CP_THREADS && (st < 0 || st > nb))
                st = nb;
            start_s[c] = st;
        }
        __syncthreads();
        const int st = start_s[tid];
        const bool valid = st >= 0;
        int en = nb;
        if (valid) {
            int c = tid + 1;
            while (start_s[c] < 0)
                c++;
            en = start_s[c];
        }
        const bool last_tile = start_s[CP_THREADS] >= nb;
        if (!__syncthreads_or(valid))
            continue;
        // ---- pass 1: the four hypotheses ----
        uint32_t lps4_0 = 0, shw_0 = 0; // table row of the LPS bin in front of the chunk
        ChunkMap m = chunkmap_identity();
        if (valid) {
            uint32_t r[4] = {510, 510, 510, 510};
            if (st > 0) {
                const uint2 t0 = rtab[(M(st - 1) >> 3) & 63];
                lps4_0 = t0.x, shw_0 = t0.y;
#pragma unroll
                for (int h = 0; h < 4; h++)
                    r[h] = cabac_range_after_lps(lps4_0, shw_0, h);
            }
            m.qmap = 0;
            const bool closing = en < nb; // bin en - 1 is the LPS bin in front of the next chunk
            const int stop = closing ? en - 1 : en;
            for (int i = st; i < stop; i++) {
                const uint32_t mm = M(i);
                const uint2 t = rtab[(mm >> 3) & 63];
#pragma unroll
                for (int h = 0; h < 4; h++) {
                    uint32_t add, pre1, sh;
                    cabac_rstep(r[h], mm, t.x, t.y, add, pre1, sh);
                    m.s[h] += pre1 + sh;
                }
            }
            if (closing) {
                const uint2 t = rtab[(M(en - 1) >> 3) & 63];
#pragma unroll
                for (int h = 0; h < 4; h++) {
                    const uint32_t q = (r[h] >> 6) & 3;
                    m.qmap |= q << (2 * h);
                    m.s[h] += (t.y >> (3 * q)) & 7;
                }
            }
        }
        // ---- scan of the chunk maps (per warp, then over the warps): true hypothesis and stream position ----
        ChunkMap run = m;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            ChunkMap o = shfl_up_map(run, off);
            if (lane >= off)
                run = chunkmap_compose(o, run);
        }
        ChunkMap ex = shfl_up_map(run, 1); // chunks of this warp in front of this one
        if (lane == 0)
            ex = chunkmap_identity();
        if (lane == 31) {
            wmap_s[warp][0] = run.qmap;
#pragma unroll
            for (int h = 0; h < 4; h++)
                wmap_s[warp][1 + h] = run.s[h];
        }
        __syncthreads();
        const uint32_t cq = carry_q, cP = carry_P;
        ChunkMap pre = chunkmap_identity(); // warps in front of this one
        for (int w2 = 0; w2 < warp; w2++) {
            ChunkMap o;
            o.qmap = wmap_s[w2][0];
#pragma unroll
            for (int h = 0; h < 4; h++)
                o.s[h] = wmap_s[w2][1 + h];
            pre = chunkmap_compose(pre, o);
        }
        ex = chunkmap_compose(pre, ex);
        const uint32_t q_in = (ex.qmap >> (2 * cq)) & 3;
        uint32_t P = cP + sel4(ex.s, cq);
        __syncthreads();
        if (tid == CP_THREADS - 1) {
            const ChunkMap tot = chunkmap_compose(ex, m);
            carry_q = (tot.qmap >> (2 * cq)) & 3;
            carry_P = cP + sel4(tot.s, cq);
        }
        __syncthreads();
        // ---- initialise the limbs this tile reaches ----
        const int hi = (int)((carry_P + 8) >> 4);
        if ((unsigned long long)hi + 2 > eb.limb_cap)
            overflow = true;
        if (overflow)
            break;
        for (int j = prev_hi + 1 + tid; j <= hi; j += CP_THREADS)
            limbs[j] = 0;
        prev_hi = hi;
        __threadfence();
        __syncthreads();
        // ---- pass 2: the true walk.  The thread's values collect in two limb registers (limb jc and jc + 1) ----
        if (valid) {
            uint32_t range = st > 0 ? cabac_range_after_lps(lps4_0, shw_0, q_in) : 510u;
            uint32_t jc = P >> 4, cur = 0, nxt = 0;
            auto adder = [&](unsigned long long j, uint32_t v) {
                if ((uint32_t)j == jc)
                    cur += v;
                else
                    nxt += v;
            };
            for (int i = st; i < en; i++) {
                const uint32_t mm = M(i);
                const uint2 t = rtab[(mm >> 3) & 63];
                uint32_t add, pre1, sh;
                cabac_rstep(range, mm, t.x, t.y, add, pre1, sh);
                P += pre1;
                if (add) {
                    const uint32_t j = P >> 4;
                    if (j != jc) { // moved on: hand the finished limb(s) over
                        if (cur)
                            atomicAdd(limbs + jc, cur);
                        if (j == jc + 1)
                            cur = nxt;
                        else {
                            if (nxt)
                                atomicAdd(limbs + jc + 1, nxt);
                            cur = 0;
                        }
                        nxt = 0;
                        jc = j;
                    }
                    limb_add(adder, P, add);
                }
                P += sh;
            }
            if (cur)
                atomicAdd(limbs + jc, cur);
            if (nxt)
                atomicAdd(limbs + jc + 1, nxt);
        }
        if (last_tile)
            break;
    }
    __threadfence();
    __syncthreads();
    // ---- carry-lookahead over the limbs (from the end of the stream to its start), stop bit, bytes ----
    const uint32_t T_end = carry_P;
    const uint32_t nbytes = (T_end + 2 + 7) >> 3;
    if (!overflow && (unsigned long long)hb + nbytes + 64 > eb.rbsp_cap)
        overflow = true;
    if (overflow) {
        if (tid == 0) {
            atomicExch(eb.error, 3);
            eb.rbsp_len[u] = 0;
        }
        return;
    }
    const int NL = prev_hi + 1;
    const uint32_t sb = T_end + 1; // stream position of the rbsp stop bit
    if (tid == 0)
        cin_s = 0;
    __syncthreads();
    for (int j0 = ((NL - 1) / CP_THREADS) * CP_THREADS; j0 >= 0; j0 -= CP_THREADS) {
        const int j = j0 + tid;
        const uint32_t x = j < NL ? __ldcg(limbs + j) : 0, xn = j + 1 < NL ? __ldcg(limbs + j + 1) : 0;
        const uint32_t w = (x & 0xffff) + (xn >> 16); // <= 0xffff + 24: single-bit carries from here on
        // lane with the higher limb index = less significant: bit 31 - lane, so carries run up an integer add
        const uint32_t G = __brev(__ballot_sync(0xffffffffu, (w >> 16) != 0));
        const uint32_t Pm = __brev(__ballot_sync(0xffffffffu, (w & 0xffff) == 0xffff));
        if (lane == 0) {
            wg_s[warp] = (uint32_t)(((unsigned long long)(G | Pm) + G) >> 32);
            wp_s[warp] = Pm == 0xffffffffu;
        }
        __syncthreads();
        // the same trick over the warps: warp w's carry in = carry out of warps w + 1 .. (higher limbs)
        const uint32_t G2 = __brev(__ballot_sync(0xffffffffu, lane < CP_WARPS && wg_s[lane])) >> (32 - CP_WARPS);
        const uint32_t P2 = __brev(__ballot_sync(0xffffffffu, lane < CP_WARPS && wp_s[lane])) >> (32 - CP_WARPS);
        const uint32_t sum2 = (G2 | P2) + G2 + cin_s; // bit k <-> warp CP_WARPS - 1 - k; bit CP_WARPS = carry out
        const uint32_t C2 = (G2 | P2) ^ G2 ^ sum2;
        const uint32_t c = (C2 >> (CP_WARPS - 1 - warp)) & 1;
        const unsigned long long sum = (unsigned long long)(G | Pm) + G + c;
        const uint32_t C = (G | Pm) ^ G ^ (uint32_t)sum; // carry into every bit
        uint32_t o = (w + ((C >> (31 - lane)) & 1)) & 0xffff;
        __syncthreads();
        if (tid == 0)
            cin_s = (sum2 >> CP_WARPS) & 1;
        // 9.3.4.5 flush: code-word bits below the stop bit are dropped, the stop bit is set
        if ((uint32_t)j > (sb >> 4))
            o = 0;
        else if ((uint32_t)j == (sb >> 4)) {
            const uint32_t k2 = sb & 15;
            o = (o & ~((1u << (16 - k2)) - 1)) | (1u << (15 - k2));
        }
        if (2u * j < nbytes)
            out[hb + 2 * j] = (uint8_t)(o >> 8);
        if (2u * j + 1 < nbytes)
            out[hb + 2 * j + 1] = (uint8_t)o;
    }
    if (tid == 0)
        eb.rbsp_len[u] = hb + nbytes;
}

// ================================================================================================
// K8 emulation prevention + NAL assembly.  Each thread owns a 64-byte chunk of a frame's RBSP:
// pass 1 counts the 0x03 bytes it must insert (order-independent rule, epb_needed), a scan gives
// chunk and frame offsets, pass 2 writes start code, NAL header and escaped payload into the packed
// output stream.
// ================================================================================================
#define EPB_CHUNK 64

// SPS + PPS bytes (host written) and which slice NALs they precede: mode 0 none, 1 the first NAL of this call
// (stream frame 0, cedar.c:1058-1061), 2 the first slice of every IDR picture (repeat_headers extension).
struct ParamSets {
    uint8_t bytes[64];
    int len, mode;
};
__device__ __forceinline__ bool has_param_sets(const ParamSets &ps, int u, int nslices, int gop_len, int first_frame_index)
{
    if (u % nslices)
        return false;
    return (ps.mode == 1 && u == 0) || (ps.mode == 2 && ((first_frame_index + u / nslices) % gop_len) == 0);
}

__device__ __forceinline__ unsigned zero_run_before(const uint8_t *p, long i)
{
    unsigned run = 0;
    for (long j = i - 1; j >= 0 && p[j] == 0; j--)
        run++;
    return run;
}

__global__ void epb_count_kernel(int nframes, const uint8_t *__restrict__ rbsp, unsigned rbsp_cap,
                                 const uint32_t *__restrict__ rbsp_len, uint32_t *__restrict__ chunk_cnt,
                                 unsigned chunks_per_frame, unsigned cblocks)
{
    int f = (int)(blockIdx.x / cblocks);
    unsigned ch = (blockIdx.x % cblocks) * blockDim.x + threadIdx.x;
    if (f >= nframes || ch >= chunks_per_frame)
        return;
    const uint8_t *p = rbsp + (size_t)f * rbsp_cap;
    long n = rbsp_len[f], b = (long)ch * EPB_CHUNK, e = b + EPB_CHUNK < n ? b + EPB_CHUNK : n;
    uint32_t cnt = 0;
    if (b < n) {
        unsigned run = zero_run_before(p, b);
        for (long i = b; i < e; i++) {
            int v = p[i];
            cnt += epb_needed(v, run);
            run = v ? 0 : run + 1;
        }
    }
    chunk_cnt[(size_t)f * chunks_per_frame + ch] = cnt;
}

// One CTA per frame: exclusive scan of its chunk counts (in place) and the frame's NAL size.
__global__ void __launch_bounds__(1024) epb_scan_kernel(int nframes, const uint32_t *__restrict__ rbsp_len,
                                                        uint32_t *chunk_cnt, unsigned chunks_per_frame,
                                                        uint32_t *__restrict__ nal_bytes, ParamSets ps, int nslices,
                                                        int gop_len, int first_frame_index)
{
    const int f = blockIdx.x;
    uint32_t *c = chunk_cnt + (size_t)f * chunks_per_frame;
    const uint32_t epb = block_exclusive_scan(c, c, (rbsp_len[f] + EPB_CHUNK - 1) / EPB_CHUNK, 0u);
    if (threadIdx.x == 0)
        nal_bytes[f] = rbsp_len[f] ? 5 + rbsp_len[f] + epb + // start code + NAL header + payload (+ SPS, PPS in front)
                                         (has_param_sets(ps, f, nslices, gop_len, first_frame_index) ? ps.len : 0)
                                   : 0;
}

// Single CTA: exclusive scan of the NAL sizes (one per slice NAL) -> offsets in the packed stream.
// frame_bytes[f] additionally counts the parameter sets that precede frame 0 (cedar.c:1058-1061).
__global__ void __launch_bounds__(1024) pack_scan_kernel(int nunits, int nslices, const uint32_t *__restrict__ nal_bytes,
                                                         unsigned prefix_bytes, unsigned long long *nal_off,
                                                         int *__restrict__ frame_bytes, unsigned long long *total,
                                                         unsigned long long out_cap, int *error)
{
    const int tid = threadIdx.x;
    const unsigned long long end_all = block_exclusive_scan(nal_bytes, nal_off, nunits, (unsigned long long)prefix_bytes);
    // bytes per picture = its slice NALs (+ the parameter sets in front of picture 0)
    for (int fr = tid; fr < nunits / nslices; fr += 1024) {
        unsigned long long b = fr == 0 ? 0 : nal_off[(size_t)fr * nslices];
        unsigned long long e = (fr + 1) * nslices < nunits ? nal_off[(size_t)(fr + 1) * nslices] : end_all;
        frame_bytes[fr] = (int)(e - b);
    }
    if (tid == 0) {
        *total = end_all;
        if (end_all > out_cap) {
            atomicExch(error, 4);
            *total = 0;
        }
    }
}

__global__ void epb_write_kernel(int nframes /* units */, int nslices, int gop_len, int first_frame_index,
                                 const uint8_t *__restrict__ rbsp, unsigned rbsp_cap,
                                 const uint32_t *__restrict__ rbsp_len, const uint32_t *__restrict__ chunk_off,
                                 unsigned chunks_per_frame, unsigned cblocks, const unsigned long long *__restrict__ nal_off,
                                 const unsigned long long *__restrict__ total, uint8_t *__restrict__ out, ParamSets ps)
{
    int f = (int)(blockIdx.x / cblocks);
    unsigned ch = (blockIdx.x % cblocks) * blockDim.x + threadIdx.x;
    if (f >= nframes || ch >= chunks_per_frame || *total == 0)
        return;
    const uint8_t *p = rbsp + (size_t)f * rbsp_cap;
    long n = rbsp_len[f], b = (long)ch * EPB_CHUNK, e = b + EPB_CHUNK < n ? b + EPB_CHUNK : n;
    if (n == 0)
        return;
    uint8_t *o = out + nal_off[f];
    if (has_param_sets(ps, f, nslices, gop_len, first_frame_index)) {
        if (ch == 0)
            for (int i = 0; i < ps.len; i++)
                o[i] = ps.bytes[i];
        o += ps.len;
    }
    if (ch == 0) {
        // cedar.c:868-881 start code + NAL header: IDR ref_idc 3 type 5, P ref_idc 2 type 1 (:987-990)
        int frame_i = ((first_frame_index + f / nslices) % gop_len) == 0;
        o[0] = 0, o[1] = 0, o[2] = 0, o[3] = 1;
        o[4] = frame_i ? 0x65 : 0x41;
    }
    if (b >= n)
        return;
    o += 5 + b + chunk_off[(size_t)f * chunks_per_frame + ch];
    unsigned run = zero_run_before(p, b);
    for (long i = b; i < e; i++) {
        int v = p[i];
        if (epb_needed(v, run))
            *o++ = 3;
        *o++ = (uint8_t)v;
        run = v ? 0 : run + 1;
    }
}

} // namespace cedar
