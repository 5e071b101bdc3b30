// GPU test harness of the entropy back end: launches the product's own CABAC kernels (cabac_resolve_kernel,
// cabac_code_kernel) and NAL assembly kernels (epb_count / epb_scan / pack_scan / epb_write) from csrc/kernels.cuh on
// caller-built inputs, the way encoder.cu launches them.  TEST ONLY (tests/test_entropy_backend.py), like
// host_harness.cpp: it is not linked into the product library.
//
// Every device buffer lies between two guard regions filled with a known byte; after the kernels ran, the whole
// allocation is copied back and the guards are compared, so an out-of-bounds write shows up as a failed call.
#include "../cedarx_h264_encoder_b200/csrc/kernels.cuh"

#include <cuda_runtime.h>

#include <cstring>
#include <vector>

using namespace cedar;

namespace {

constexpr size_t GUARD = 4096;      // bytes on each side; a multiple of 256 keeps the payload as aligned as cudaMalloc's
constexpr uint8_t GUARD_BYTE = 0xa5;

// Error codes of the entry points (the kernels' own error word is returned separately).
enum { CG_OK = 0, CG_CUDA = -1, CG_ARGS = -2, CG_GUARD = -100 /* - buffer index */ };

struct Guarded {
    uint8_t *base = nullptr;
    size_t bytes = 0;
    void *ptr() const { return base + GUARD; }
};

struct Arena {
    std::vector<Guarded> bufs;
    bool failed = false;
    ~Arena()
    {
        for (auto &b : bufs)
            cudaFree(b.base);
    }
    // payload of `bytes` bytes, filled with `init` (or with `fill` when init is null)
    template <class T> T *alloc(size_t bytes, const void *init, uint8_t fill = 0xcd)
    {
        Guarded g;
        g.bytes = bytes;
        if (cudaMalloc(&g.base, bytes + 2 * GUARD) != cudaSuccess) {
            failed = true;
            return nullptr;
        }
        bufs.push_back(g);
        if (cudaMemset(g.base, GUARD_BYTE, bytes + 2 * GUARD) != cudaSuccess ||
            (init ? cudaMemcpy(g.ptr(), init, bytes, cudaMemcpyHostToDevice)
                  : cudaMemset(g.ptr(), fill, bytes)) != cudaSuccess)
            failed = true;
        return (T *)g.ptr();
    }
    // copies every payload's guards back: 0 if intact, else CG_GUARD - (index of the first damaged buffer)
    int check_guards() const
    {
        std::vector<uint8_t> h(GUARD);
        for (size_t i = 0; i < bufs.size(); i++)
            for (int side = 0; side < 2; side++) {
                const uint8_t *src = side ? bufs[i].base + GUARD + bufs[i].bytes : bufs[i].base;
                if (cudaMemcpy(h.data(), src, GUARD, cudaMemcpyDeviceToHost) != cudaSuccess)
                    return CG_CUDA;
                for (size_t k = 0; k < GUARD; k++)
                    if (h[k] != GUARD_BYTE)
                        return CG_GUARD - (int)i;
            }
        return CG_OK;
    }
};

int finish(Arena &a, cudaStream_t st)
{
    const bool ok = cudaStreamSynchronize(st) == cudaSuccess && cudaGetLastError() == cudaSuccess;
    cudaStreamDestroy(st);
    if (!ok || a.failed)
        return CG_CUDA;
    return a.check_guards();
}

} // namespace

extern "C" {

// CABAC back end on one stream: cabac_resolve_kernel, then cabac_code_kernel, one CTA per (lane, slice) as in
// encoder.cu.  Units u = frame * nslices + slice, U = nframes * nslices of them; the lanes of `Step` choose the frames
// coded, (gop_pos0 + frame) % gop_len == 0 makes a frame an I frame.
//   pool[pool_len]           bins (in) -> the resolver's records in place of every coded bin (out)
//   bins_off / bins_len [U]  where each unit's bins lie in the pool
//   hdr_bits / hdr_nbits [U] slice header bits
//   rbsp [U * rbsp_cap]      out; rbsp_len [U] in: initial values (a sentinel), out: as the kernels left them
//   ctx_hist [464] or null   in / out: the resolver adds every context's regular bin count
//   *error                   the kernels' sticky error word (0 in)
// Returns 0, CG_CUDA, CG_ARGS, or CG_GUARD - i when the guards of device buffer i were overwritten.
int cg_cabac_backend(uint16_t *pool, unsigned long long pool_len, int nslices, int qp, int gop_len, int gop_pos0,
                     int nlanes, int frame0, int lane_stride, int nframes, const unsigned long long *bins_off,
                     const uint32_t *bins_len, const unsigned long long *hdr_bits, const int *hdr_nbits,
                     unsigned rbsp_cap, unsigned long long limb_cap, uint8_t *rbsp, uint32_t *rbsp_len,
                     unsigned long long *ctx_hist, int *error)
{
    if (nslices < 1 || nlanes < 1 || nframes < 1 || gop_len < 1 || pool_len == 0 || rbsp_cap == 0 || limb_cap == 0)
        return CG_ARGS;
    const size_t U = (size_t)nframes * nslices, ctas = (size_t)nlanes * nslices;
    if (cudaFuncSetAttribute(cabac_code_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CP_SMEM_BYTES) != cudaSuccess ||
        cudaFuncSetAttribute(cabac_resolve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, RES_SMEM_BYTES) != cudaSuccess)
        return CG_CUDA;
    Arena a;
    EntropyBufs eb;
    memset(&eb, 0, sizeof(eb));
    eb.bins = a.alloc<uint16_t>(pool_len * 2, pool);
    eb.bins_cap = pool_len;
    eb.bins_off = a.alloc<unsigned long long>(U * 8, bins_off);
    eb.bins_len = a.alloc<uint32_t>(U * 4, bins_len);
    eb.hdr_bits = a.alloc<unsigned long long>(U * 8, hdr_bits);
    eb.hdr_nbits = a.alloc<int>(U * 4, hdr_nbits);
    eb.rbsp = a.alloc<uint8_t>(U * rbsp_cap, nullptr);
    eb.rbsp_cap = rbsp_cap;
    eb.rbsp_len = a.alloc<uint32_t>(U * 4, rbsp_len);
    eb.limbs = a.alloc<uint32_t>(ctas * limb_cap * 4, nullptr); // stale contents: the coder initialises what it uses
    eb.limb_cap = limb_cap;
    eb.error = a.alloc<int>(4, error);
    unsigned long long *d_hist = ctx_hist ? a.alloc<unsigned long long>(464 * 8, ctx_hist) : nullptr;
    if (a.failed)
        return CG_CUDA;
    Geom g;
    memset(&g, 0, sizeof(g));
    g.nslices = nslices;
    g.qp = qp;
    const Step s{nlanes, frame0, lane_stride, nframes};
    cudaStream_t st;
    if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess)
        return CG_CUDA;
    cabac_resolve_kernel<<<(unsigned)ctas, RES_THREADS, RES_SMEM_BYTES, st>>>(g, s, gop_len, gop_pos0, eb, d_hist);
    cabac_code_kernel<<<(unsigned)ctas, CP_THREADS, CP_SMEM_BYTES, st>>>(g, s, eb);
    int r = finish(a, st);
    if (r == CG_OK &&
        (cudaMemcpy(pool, eb.bins, pool_len * 2, cudaMemcpyDeviceToHost) != cudaSuccess ||
         cudaMemcpy(rbsp, eb.rbsp, U * rbsp_cap, cudaMemcpyDeviceToHost) != cudaSuccess ||
         cudaMemcpy(rbsp_len, eb.rbsp_len, U * 4, cudaMemcpyDeviceToHost) != cudaSuccess ||
         cudaMemcpy(error, eb.error, 4, cudaMemcpyDeviceToHost) != cudaSuccess ||
         (ctx_hist && cudaMemcpy(ctx_hist, d_hist, 464 * 8, cudaMemcpyDeviceToHost) != cudaSuccess)))
        r = CG_CUDA;
    return r;
}

// NAL assembly of `nunits` slice NALs with encoder.cu's grid arithmetic: epb_count -> epb_scan -> pack_scan ->
// epb_write.  rbsp [nunits * rbsp_cap] and rbsp_len [nunits] are the RBSP units; ps_* the parameter-set bytes (at most
// 64) and mode (0 none, 1 before unit 0, 2 before the first slice of every IDR picture).  Out: out [out_cap] (the packed
// stream; bytes the kernels do not write keep their initial values, which are copied in), nal_off [nunits],
// frame_bytes [nunits / nslices], *total, *error (0 in).  Returns as cg_cabac_backend.
int cg_nal_assembly(const uint8_t *rbsp, unsigned rbsp_cap, const uint32_t *rbsp_len, int nunits, int nslices,
                    int gop_len, int first_frame_index, const uint8_t *ps_bytes, int ps_len, int ps_mode,
                    unsigned long long out_cap, uint8_t *out, unsigned long long *nal_off, int *frame_bytes,
                    unsigned long long *total, int *error)
{
    if (nunits < 1 || nslices < 1 || nunits % nslices || gop_len < 1 || rbsp_cap == 0 || out_cap == 0 || ps_len < 0 ||
        ps_len > 64)
        return CG_ARGS;
    const unsigned cpf = (rbsp_cap + EPB_CHUNK - 1) / EPB_CHUNK, cblocks = (cpf + 255) / 256;
    const int nfr = nunits / nslices;
    Arena a;
    const uint8_t *d_rbsp = a.alloc<uint8_t>((size_t)nunits * rbsp_cap, rbsp);
    const uint32_t *d_len = a.alloc<uint32_t>((size_t)nunits * 4, rbsp_len);
    uint32_t *d_chunk = a.alloc<uint32_t>((size_t)cpf * nunits * 4, nullptr);
    uint32_t *d_nal_bytes = a.alloc<uint32_t>((size_t)nunits * 4, nullptr);
    unsigned long long *d_nal_off = a.alloc<unsigned long long>((size_t)nunits * 8, nullptr);
    int *d_frame_bytes = a.alloc<int>((size_t)nfr * 4, nullptr);
    unsigned long long *d_total = a.alloc<unsigned long long>(8, nullptr);
    uint8_t *d_out = a.alloc<uint8_t>(out_cap, out);
    int *d_error = a.alloc<int>(4, error);
    if (a.failed)
        return CG_CUDA;
    ParamSets ps;
    memset(&ps, 0, sizeof(ps));
    if (ps_len)
        memcpy(ps.bytes, ps_bytes, (size_t)ps_len);
    ps.len = ps_len;
    ps.mode = ps_mode;
    cudaStream_t st;
    if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess)
        return CG_CUDA;
    epb_count_kernel<<<(unsigned)nunits * cblocks, 256, 0, st>>>(nunits, d_rbsp, rbsp_cap, d_len, d_chunk, cpf, cblocks);
    epb_scan_kernel<<<nunits, 1024, 0, st>>>(nunits, d_len, d_chunk, cpf, d_nal_bytes, ps, nslices, gop_len,
                                             first_frame_index);
    pack_scan_kernel<<<1, 1024, 0, st>>>(nunits, nslices, d_nal_bytes, 0u, d_nal_off, d_frame_bytes, d_total, out_cap,
                                         d_error);
    epb_write_kernel<<<(unsigned)nunits * cblocks, 256, 0, st>>>(nunits, nslices, gop_len, first_frame_index, d_rbsp,
                                                                 rbsp_cap, d_len, d_chunk, cpf, cblocks, d_nal_off,
                                                                 d_total, d_out, ps);
    int r = finish(a, st);
    if (r == CG_OK &&
        (cudaMemcpy(out, d_out, out_cap, cudaMemcpyDeviceToHost) != cudaSuccess ||
         cudaMemcpy(nal_off, d_nal_off, (size_t)nunits * 8, cudaMemcpyDeviceToHost) != cudaSuccess ||
         cudaMemcpy(frame_bytes, d_frame_bytes, (size_t)nfr * 4, cudaMemcpyDeviceToHost) != cudaSuccess ||
         cudaMemcpy(total, d_total, 8, cudaMemcpyDeviceToHost) != cudaSuccess ||
         cudaMemcpy(error, d_error, 4, cudaMemcpyDeviceToHost) != cudaSuccess))
        r = CG_CUDA;
    return r;
}
}
