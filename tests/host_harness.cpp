// CPU unit-test harness: compiles the product's per-macroblock entropy logic (entropy.cuh,
// h264_core.cuh) as ordinary C++ and drives it the way the CUDA kernels do (count pass, prefix sum,
// scatter pass; binarise then serial arithmetic coder; parallel-rule emulation prevention).
// TEST ONLY: it lets `pytest -m "not gpu"` compare this logic with the oracle without a GPU.
// It is not linked into the product library and does not link the oracle.
#include "../cedarx_h264_encoder_b200/csrc/entropy.cuh"

#include <algorithm>
#include <cstring>
#include <vector>

using namespace cedar;

extern "C" {

// One slice (macroblock rows [row0, row1) of a picture whose slices are srows rows tall) through the
// count / prefix-sum / scatter passes.  Returns RBSP length in bytes (header bits + slice data + trailing
// bits, byte aligned).
long hh_cavlc_slice(const void *mbi, const uint8_t *nnz, const int16_t *coef, int mbw, int mbh, int srows, int slice,
                    int frame_i, uint64_t hdr_bits, int hdr_nbits, uint8_t *out, long cap, const uint8_t *i4)
{
    FrameSyntax fs{(const MbInfo *)mbi, nnz, coef, mbw, mbh, srows, i4};
    const int per = slice_items_per(fs), nitems = mbw * mbh + (mbh + srows - 1) / srows;
    const int j0 = slice * per, j1 = per * (slice + 1) < nitems ? per * (slice + 1) : nitems;
    std::vector<unsigned long long> off(j1 - j0 + 1);
    unsigned long long pos = (unsigned long long)hdr_nbits;
    for (int j = j0; j < j1; j++) {
        SliceItem it = slice_item(fs, j);
        if (it.slice != slice || it.is_first != (j == j0) || it.is_end != (j == j1 - 1))
            return -3;
        BitCount c;
        int run = frame_i ? 0 : skip_run_before(fs, it.mb, it.first_mb);
        if (it.is_end)
            cavlc_end(c, run);
        else if (fs.mbi[it.mb].type != MB_PSKIP)
            cavlc_mb(c, fs, it.mb, frame_i, run);
        off[j - j0] = pos;
        pos += c.n;
    }
    long bytes = (long)((pos + 7) >> 3);
    if (bytes > cap)
        return -1;
    std::vector<uint32_t> buf((size_t)(bytes + 8) / 4 + 2, 0);
    {
        BitScatter s(buf.data(), 0);
        if (hdr_nbits > 32)
            s.put((uint32_t)(hdr_bits >> 32), hdr_nbits - 32);
        s.put((uint32_t)hdr_bits, hdr_nbits > 32 ? 32 : hdr_nbits);
        s.flush();
    }
    // scatter in reverse order to show the order does not matter
    for (int j = j1 - 1; j >= j0; j--) {
        SliceItem it = slice_item(fs, j);
        int run = frame_i ? 0 : skip_run_before(fs, it.mb, it.first_mb);
        if (!it.is_end && fs.mbi[it.mb].type == MB_PSKIP)
            continue;
        BitScatter s(buf.data(), off[j - j0]);
        if (it.is_end)
            cavlc_end(s, run);
        else
            cavlc_mb(s, fs, it.mb, frame_i, run);
        s.flush();
    }
    memcpy(out, buf.data(), (size_t)bytes);
    return bytes;
}

// The bins of one slice (macroblock rows [row0, row1) of a picture whose slices are srows rows tall) through the
// count / prefix-sum / write passes.  Returns the bin count; the bins are written only if they fit in cap.
long hh_cabac_bins(const void *mbi, const uint8_t *nnz, const int16_t *coef, int mbw, int mbh, int srows, int slice,
                   int frame_i, uint16_t *bins, long cap, const uint8_t *i4)
{
    FrameSyntax fs{(const MbInfo *)mbi, nnz, coef, mbw, mbh, srows, i4};
    const int row0 = slice * srows, row1 = row0 + srows < mbh ? row0 + srows : mbh;
    const int mb0 = row0 * mbw, nmb = (row1 - row0) * mbw;
    std::vector<size_t> off(nmb + 1);
    size_t total = 0;
    for (int i = 0; i < nmb; i++) {
        BinCount c;
        cabac_mb(c, fs, mb0 + i, frame_i);
        off[i] = total;
        total += c.n;
    }
    if ((long)total > cap)
        return (long)total;
    for (int i = nmb - 1; i >= 0; i--) {
        BinWrite w(bins + off[i]);
        cabac_mb(w, fs, mb0 + i, frame_i);
    }
    return (long)total;
}

// A slice's bins (ending with terminate(1)) through the serial three-stage coder and, checked against it byte for
// byte, the parallel formulation of cabac_code_kernel emulated with chunk_bins bins per chunk.  Returns the RBSP length
// in bytes (header bits + cabac_alignment_one_bits + slice data + stop bit, byte aligned) or a negative code.
long hh_cabac_code_bins(const uint16_t *bins, long n, int frame_i, int qp, uint64_t hdr_bits, int hdr_nbits, uint8_t *out,
                        long cap, int chunk_bins)
{
    const size_t total = (size_t)n;
    // header bits followed by cabac_alignment_one_bit up to the byte boundary
    int hb = (hdr_nbits + 7) >> 3;
    unsigned long long h = (hdr_bits << (hb * 8 - hdr_nbits)) | ((1ull << (hb * 8 - hdr_nbits)) - 1);
    for (int i = 0; i < hb; i++)
        out[i] = (uint8_t)(h >> (8 * (hb - 1 - i)));
    // pre-state resolution (sequential here; per-context parallel in cabac_kernel), then the coder
    CabacTables tab;
    tab.build(0, 1);
    uint32_t state[460];
    for (int i = 0; i < 460; i++)
        state[i] = cabac_init_state(i, frame_i, qp);
    std::vector<uint8_t> pre(total + 1, 0);
    for (size_t i = 0; i < total; i++) {
        uint16_t b = bins[i];
        if (!(b & (BIN_BYPASS | BIN_TERM))) {
            int ctx = b & 0x3ff;
            pre[i] = (uint8_t)state[ctx];
            state[ctx] = cabac_next_state(tab, state[ctx], (b >> 15) & 1);
        }
    }
    // stage 2 (range recurrence -> interval steps) and stage 3 (low recurrence -> bytes)
    CabacRange rc;
    std::vector<uint32_t> steps(total + 1);
    uint32_t flat_range = 510;
    for (size_t i = 0; i < total; i++) {
        uint32_t lps4 = tab.lpsw[(pre[i] >> 1) & 63], meta = cabac_stage_meta(bins[i], pre[i], tab);
        steps[i] = rc.step(lps4, meta);
        if (cabac_range_step_flat(flat_range, lps4, meta) != steps[i] || (flat_range != rc.range && i + 1 < total))
            return -2; // the branch-free variant must agree step by step
    }
    CabacBytes c;
    std::vector<uint8_t> serial_out(cap + 16);
    c.out = serial_out.data();
    for (size_t i = 0; i < total; i++) {
        if ((long)(hb + c.pos + 8) > cap)
            return -1;
        if (i + 1 < total)
            c.step_fast(steps[i]);
        else
            c.step(steps[i]);
    }
    // ---- the parallel formulation the GPU runs (cabac_code_kernel), emulated chunk by chunk ----
    const long nb = (long)total;
    std::vector<uint16_t> meta(total + 1);
    for (long i = 0; i < nb; i++)
        meta[i] = cabac_meta(bins[i], pre[i]);
    const int K = chunk_bins > 0 ? chunk_bins : 62;
    const long nchunks = (nb + K - 1) / K;
    std::vector<long> start(nchunks + 1, -1);
    for (long k = 0; k < nchunks; k++) {
        if (k == 0) {
            start[0] = 0;
            continue;
        }
        for (long i = k * K; i < std::min(nb, (k + 1) * K); i++)
            if (cabac_meta_is_lps(meta[i])) {
                start[k] = i + 1 < nb ? i + 1 : -1; // an LPS in the very last position opens no chunk
                break;
            }
    }
    start[nchunks] = nb;
    auto next_start = [&](long k) {
        for (long j = k + 1; j <= nchunks; j++)
            if (start[j] >= 0)
                return start[j];
        return nb;
    };
    // pass 1: four hypotheses per chunk
    std::vector<ChunkMap> maps(nchunks, chunkmap_identity());
    for (long k = 0; k < nchunks; k++) {
        if (start[k] < 0)
            continue;
        long st = start[k], en = next_start(k);
        uint32_t r[4];
        ChunkMap m;
        m.qmap = 0;
        for (int h = 0; h < 4; h++) {
            m.s[h] = 0;
            if (st == 0)
                r[h] = 510;
            else {
                uint32_t ps = (meta[st - 1] >> 3) & 63;
                r[h] = cabac_range_after_lps(tab.lpsw[ps], tab.shw[ps], h);
            }
        }
        const bool closing_lps = en < nb; // bin en - 1 is the LPS bin that opens the next chunk
        for (long i = st; i < (closing_lps ? en - 1 : en); i++) {
            uint32_t ps = (meta[i] >> 3) & 63;
            for (int h = 0; h < 4; h++) {
                uint32_t add, pre1, sh;
                cabac_rstep(r[h], meta[i], tab.lpsw[ps], tab.shw[ps], add, pre1, sh);
                m.s[h] += pre1 + sh;
            }
        }
        if (closing_lps) {
            uint32_t ps = (meta[en - 1] >> 3) & 63;
            if (!cabac_meta_is_lps(meta[en - 1]))
                return -4;
            for (int h = 0; h < 4; h++) {
                uint32_t q = (r[h] >> 6) & 3;
                m.qmap |= q << (2 * h);
                m.s[h] += (tab.shw[ps] >> (3 * q)) & 7;
            }
        }
        maps[k] = m;
    }
    // scan (sequential here): true hypothesis and stream position of every chunk
    std::vector<uint32_t> qin(nchunks, 0);
    std::vector<unsigned long long> pbase(nchunks, 0);
    ChunkMap acc = chunkmap_identity();
    for (long k = 0; k < nchunks; k++) {
        qin[k] = acc.qmap & 3; // hypothesis 0 of the running composition: chunk 0 ignores its input
        pbase[k] = acc.s[0];
        acc = chunkmap_compose(acc, maps[k]);
    }
    const unsigned long long T_end = acc.s[0];
    // pass 2: true walk + limb accumulation
    std::vector<uint32_t> limbs((T_end + 8) / 16 + 3, 0);
    auto adder = [&](unsigned long long j, uint32_t v) { limbs[j] += v; };
    for (long k = nchunks - 1; k >= 0; k--) { // any order
        if (start[k] < 0)
            continue;
        long st = start[k], en = next_start(k);
        uint32_t range = 510;
        if (st > 0) {
            uint32_t ps = (meta[st - 1] >> 3) & 63;
            range = cabac_range_after_lps(tab.lpsw[ps], tab.shw[ps], qin[k]);
        }
        unsigned long long P = pbase[k];
        for (long i = st; i < en; i++) {
            uint32_t ps = (meta[i] >> 3) & 63, add, pre1, sh;
            cabac_rstep(range, meta[i], tab.lpsw[ps], tab.shw[ps], add, pre1, sh);
            P += pre1;
            if (add)
                limb_add(adder, P, add);
            P += sh;
        }
        if (P != (k + 1 < nchunks ? [&] { for (long j = k + 1; j < nchunks; j++) if (start[j] >= 0) return pbase[j]; return T_end; }() : T_end))
            return -5;
    }
    // carry resolution (two-step, as the kernel does it) + stop bit
    const long NL = (long)((T_end + 8) >> 4) + 1;
    std::vector<uint32_t> w(NL + 1, 0);
    for (long j = 0; j < NL; j++)
        w[j] = (limbs[j] & 0xffff) + (limbs[j + 1] >> 16);
    uint32_t carry = 0;
    std::vector<uint16_t> o16(NL);
    for (long j = NL - 1; j >= 0; j--) {
        uint32_t v = w[j] + carry;
        o16[j] = (uint16_t)v;
        carry = v >> 16;
    }
    if (carry)
        return -6;
    const unsigned long long sb = T_end + 1; // stream position of the stop bit
    const long nbytes = (long)((T_end + 2 + 7) >> 3);
    for (long j = 0; j < NL; j++) {
        if ((unsigned long long)j > (sb >> 4))
            o16[j] = 0;
        else if ((unsigned long long)j == (sb >> 4)) {
            uint32_t k2 = (uint32_t)sb & 15;
            o16[j] = (uint16_t)((o16[j] & ~((1u << (16 - k2)) - 1)) | (1u << (15 - k2)));
        }
    }
    if (nbytes != (long)c.pos)
        return -7;
    for (long i = 0; i < nbytes; i++) {
        uint8_t v = (uint8_t)(i & 1 ? o16[i >> 1] & 0xff : o16[i >> 1] >> 8);
        if (v != serial_out[i])
            return -8;
        out[hb + i] = v;
    }
    return hb + (long)c.pos;
}

long hh_cabac_slice(const void *mbi, const uint8_t *nnz, const int16_t *coef, int mbw, int mbh, int srows, int slice,
                    int frame_i, int qp, uint64_t hdr_bits, int hdr_nbits, uint8_t *out, long cap, int chunk_bins,
                    const uint8_t *i4)
{
    const long n = hh_cabac_bins(mbi, nnz, coef, mbw, mbh, srows, slice, frame_i, nullptr, 0, i4);
    std::vector<uint16_t> bins(n + 1);
    hh_cabac_bins(mbi, nnz, coef, mbw, mbh, srows, slice, frame_i, bins.data(), n, i4);
    return hh_cabac_code_bins(bins.data(), n, frame_i, qp, hdr_bits, hdr_nbits, out, cap, chunk_bins);
}

// Emulation prevention with the order-independent rule used by the GPU kernel.
long hh_epb(const uint8_t *in, long n, uint8_t *out, long cap)
{
    long o = 0;
    for (long i = 0; i < n; i++) {
        unsigned run = 0;
        for (long j = i - 1; j >= 0 && in[j] == 0; j--)
            run++;
        if (epb_needed(in[i], run)) {
            if (o >= cap)
                return -1;
            out[o++] = 3;
        }
        if (o >= cap)
            return -1;
        out[o++] = in[i];
    }
    return o;
}

int hh_sizeof_mbinfo() { return (int)sizeof(MbInfo); }

// Property the range stage relies on: on the MPS path the interval never needs more than a one-bit
// renormalisation (range - rangeTabLPS >= 128 for every state and every range of the quantiser cell).
int hh_mps_renorm_at_most_one()
{
    for (int s = 0; s < 64; s++)
        for (int range = 256; range <= 510; range++)
            if (range - (int)h264_range_lps[s][(range >> 6) & 3] < 128)
                return 0;
    return 1;
}
}
