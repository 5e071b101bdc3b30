"""The entropy back end on its own: the CUDA kernels cabac_resolve_kernel + cabac_code_kernel (bins -> RBSP) and
epb_count / epb_scan / pack_scan / epb_write (RBSP -> packed NAL units), launched by tests/cabac_gpu_harness.cu on
bin sequences and RBSP units built to reach their tile, alignment and carry edges, against the golden model's
spec-literal arithmetic coder (gm_cabac_code_bins) and a plain Python packer.  The CPU tests check the same sequences
against the host build of the product's coder (serial and chunked parallel formulation) and that every family of
sequences has the property it exists for."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from common import content
from test_entropy_host import to_product_layout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "cedarx_h264_encoder_b200", "csrc")
HARNESS_SRC = os.path.join(ROOT, "tests", "cabac_gpu_harness.cu")
HARNESS_SO = os.path.join(ROOT, "tests", "libcabac_gpu_harness.so")
NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"

BIN_BYPASS, BIN_TERM, BIN_VAL = 1 << 10, 1 << 11, 1 << 15
END = BIN_TERM | BIN_VAL  # end_of_slice_flag = 1: the last bin of every slice, and only there
NCTX = 460
RES_TILE = 4096           # bins per tile of cabac_resolve_kernel
CP_TB = 512 * 62          # bins per tile of cabac_code_kernel (CP_THREADS chunks of CP_K bins)
HOT = 227                 # the context of the "hot" families
# transIdxLPS (H.264 Table 9-45)
NEXT_LPS = [0, 0, 1, 2, 2, 4, 4, 5, 6, 7, 8, 9, 9, 11, 11, 12, 13, 13, 15, 15, 16, 16, 18, 18, 19, 19, 21, 21, 22, 22, 23,
            24, 24, 25, 26, 26, 27, 27, 28, 29, 29, 30, 30, 30, 31, 32, 32, 33, 33, 33, 34, 34, 35, 35, 35, 36, 36, 36, 37,
            37, 37, 38, 38, 63]

LENGTHS = [1, 2, 3, 4, 5, 31, 32, 33, 4095, 4096, 4097, 8191, 8192, 8193, 31743, 31744, 31745, 31806, 31807, 63487,
           63488, 63489, 250000]
FAMILIES = ["uniform", "hot_mps", "hot_lps", "mps_only", "sparse_lps", "lps_heavy", "alternating", "carry", "natural"]
CARRY_RUNS = [(600, 1), (9000, 0), (70000, 1), (600, 0), (9000, 1), (70000, 0)]  # (outstanding bits, ended by a carry)


# ---------------------------------------------------------------------------------------------------------------------
# bin families
# ---------------------------------------------------------------------------------------------------------------------
def carry_segment(run, carry):
    """Bypass bins at range 510 from any codILow: nine 0s take low to 0.  With a carry: seven 1s take low to 258, every
    bin of the cycle 0,1,1,1,1,1,1,1 adds an outstanding bit and returns to 258, a 1 there carries into the run.
    Without: eight 1s take low to 2, every further 1 is outstanding, a 0 ends the run."""
    if carry:
        bits = [0] * 9 + [1] * 7 + [0, 1, 1, 1, 1, 1, 1, 1] * (run // 8) + [1]
    else:
        bits = [0] * 9 + [1] * 8 + [1] * run + [0]
    return np.array([BIN_BYPASS | (BIN_VAL if b else 0) for b in bits], np.uint16)


def init_states(oracle, frame_i, qp):
    """Initial state (pStateIdx << 1 | valMPS) of every context: the reference's pre-state of each context's first bin."""
    probe = np.append(np.arange(NCTX, dtype=np.uint16), np.uint16(END))
    return oracle.cabac_code_bins(probe, frame_i, qp)[1][:NCTX].astype(np.int64)


def simulate_values(ctx, regular, lps_prob, forced_lps, init):
    """Values of the regular bins such that bin i is coded as an LPS with probability lps_prob[i] (or surely where
    forced_lps[i]): tracks every context's state with the standard's transitions."""
    state = init.tolist()
    vals = np.zeros(ctx.size, np.uint16)
    draws = np.random.default_rng(int(ctx.size) * 7 + 1).random(ctx.size)
    for i in np.flatnonzero(regular).tolist():
        c = int(ctx[i])
        s = state[c]
        p, m = s >> 1, s & 1
        lps = forced_lps[i] or draws[i] < lps_prob[i]
        vals[i] = m ^ lps
        state[c] = ((NEXT_LPS[p] << 1) | (m ^ (p == 0))) if lps else ((min(p + 1, 62) << 1) | m)
    return vals


def make_bins(family, n, frame_i, qp, oracle, natural):
    """n bins of one family: contexts 0..459 only, exactly one end_of_slice_flag = 1, the last bin."""
    rng = np.random.default_rng([FAMILIES.index(family), n, frame_i, qp])
    m = n - 1  # bins in front of the terminating one
    init = init_states(oracle, frame_i, qp)
    if family == "carry":
        segs, k, have = [], 0, 0
        while have < m:
            segs.append(carry_segment(*CARRY_RUNS[k % len(CARRY_RUNS)]))
            have += segs[-1].size
            k += 1
        body = np.concatenate(segs)[:m] if segs else np.zeros(0, np.uint16)
    elif family == "natural":
        body = np.resize(natural, m)
    elif family == "alternating":  # a run of 0s and 1s alternating in three contexts: LPS bins everywhere
        body = ((np.arange(m) % 3) + 11 + (BIN_VAL * ((np.arange(m) // 3) % 2))).astype(np.uint16)
    else:
        u = rng.random(m)
        bypass_share = {"uniform": 0.10, "hot_mps": 0.03, "hot_lps": 0.03}.get(family, 0.08)
        bypass = u < bypass_share
        term0 = (u >= bypass_share) & (u < bypass_share + 0.02) if family == "uniform" else np.zeros(m, bool)
        regular = ~bypass & ~term0
        ctx = rng.integers(0, NCTX, m)
        if family in ("hot_mps", "hot_lps"):
            ctx = np.where(rng.random(m) < 0.97, HOT, ctx)
            whole = slice(RES_TILE, 2 * RES_TILE)  # the second resolver tile: one context, no other bin
            ctx[whole], regular[whole], bypass[whole] = HOT, True, False
        if family == "uniform":
            vals = rng.integers(0, 2, m).astype(np.uint16)
        else:
            p = {"hot_mps": 0.03, "hot_lps": 0.7, "mps_only": 0.0, "sparse_lps": 0.0, "lps_heavy": 0.9}[family]
            forced = np.zeros(m, bool)
            if family == "sparse_lps":  # one LPS bin every 40 009 bins: whole coder tiles without a chunk start
                forced[40009::40009] = True
                regular[40009::40009] = True
                bypass[40009::40009] = False
            if family == "lps_heavy":  # an LPS bin at the last position of every coder tile and as the last regular bin
                forced[CP_TB - 1::CP_TB] = True
                regular[CP_TB - 1::CP_TB] = True
                bypass[CP_TB - 1::CP_TB] = False
                if m:
                    forced[m - 1] = regular[m - 1] = True
                    bypass[m - 1] = False
            vals = simulate_values(ctx, regular, np.full(m, p), forced, init)
            vals[bypass] = rng.integers(0, 2, int(bypass.sum()))
        body = np.where(regular, ctx, np.where(bypass, BIN_BYPASS, BIN_TERM)).astype(np.uint16)
        body |= np.where(regular | bypass, vals, 0).astype(np.uint16) * BIN_VAL
    return np.append(body.astype(np.uint16), np.uint16(END))


def natural_bins(oracle, hh):
    """The product's binarisation of noise at QP 1 and synth at QP 24, 176x144, I and P frames, without the
    end_of_slice_flag = 1 of each slice."""
    w, h = 176, 144
    out = []
    for kind, qp in (("noise", 1), ("synth", 24)):
        enc = oracle.Encoder(oracle.make_config(w, h, qp=qp, gop=2, cabac=1, me_range=8))
        for t in range(2):
            enc.encode(*content(kind, w, h, t))
            mbi, nnz, coef, i4 = to_product_layout(enc.mbs())
            fi = int(enc.frame_is_i())
            args = (mbi.ctypes.data, nnz.ctypes.data, coef.ctypes.data, w // 16, h // 16, h // 16, 0, fi)
            nb = hh.hh_cabac_bins(*args, None, 0, i4.ctypes.data)
            bins = np.zeros(nb, np.uint16)
            assert hh.hh_cabac_bins(*args, bins.ctypes.data, nb, i4.ctypes.data) == nb
            assert bins[-1] == END
            out.append(bins[:-1])
        enc.close()
    return np.concatenate(out)


@pytest.fixture(scope="module")
def hh(harness):
    harness.hh_cabac_bins.restype = C.c_long
    harness.hh_cabac_bins.argtypes = [C.c_void_p] * 3 + [C.c_int] * 5 + [C.c_void_p, C.c_long, C.c_void_p]
    harness.hh_cabac_code_bins.restype = C.c_long
    harness.hh_cabac_code_bins.argtypes = [C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_void_p,
                                           C.c_long, C.c_int]
    return harness


@pytest.fixture(scope="module")
def gen(oracle, hh):
    natural = natural_bins(oracle, hh)
    cache = {}

    def g(family, n, frame_i=1, qp=24):
        key = (family, n, frame_i, qp)
        if key not in cache:
            cache[key] = make_bins(family, n, frame_i, qp, oracle, natural)
        return cache[key]
    return g


def header(k):
    """Slice-header bits of unit k: assorted lengths, byte aligned or not."""
    nbits = [13, 24, 40, 57, 62, 1, 8, 33][k % 8]
    return int(np.random.default_rng(k + 1000).integers(0, 1 << nbits, dtype=np.uint64)), nbits


def records(bins, pre):
    """cabac_meta(bin, pre-state): what the resolver leaves in place of every bin."""
    b = bins.astype(np.int64)
    pre = pre.astype(np.int64)
    special, v = (b >> 10) & 3, (b >> 15) & 1
    return np.where(special != 0, v | (special << 1), ((pre >> 1) << 3) | (v ^ (pre & 1))).astype(np.uint16)


def case_params(n):
    """Picture type and QP of the family x length cases: all three QPs and both types over the lengths."""
    k = LENGTHS.index(n)
    return 1 - k % 2, (24, 47, 1)[k % 3]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the golden model's coder, the host build of the product's coder, and the families' properties
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", LENGTHS)
@pytest.mark.parametrize("family", FAMILIES)
def test_host_parallel_coder_matches_golden_coder(oracle, hh, gen, family, n):
    """hh_cabac_code_bins checks its chunked parallel formulation against its serial coder byte for byte; both must
    equal the spec-literal coder, for chunks of 62 (the kernel's), 7 and 1000 bins."""
    frame_i, qp = case_params(n)
    bins = gen(family, n, frame_i, qp)
    hb, hn = header(n)
    want = oracle.cabac_code_bins(bins, frame_i, qp, hb, hn)[0]
    for chunk in (62, 7, 1000):
        out = np.zeros(len(want) + 4096, np.uint8)
        r = hh.hh_cabac_code_bins(bins.ctypes.data, bins.size, frame_i, qp, hb, hn, out.ctypes.data, out.size, chunk)
        assert r == len(want), (family, n, chunk, r)
        assert out[:r].tobytes() == want, (family, n, chunk)


def test_golden_bin_coder_equals_the_golden_encoder(oracle, hh):
    """gm_cabac_code_bins on the product's bins of a frame gives the slice RBSP the golden encoder itself wrote."""
    import avdec
    w, h = 176, 144
    enc = oracle.Encoder(oracle.make_config(w, h, qp=20, gop=2, cabac=1, me_range=8))
    for t in range(2):
        nals = [nal for ty, nal in avdec.split_nals(enc.encode(*content("synth", w, h, t))) if ty in (1, 5)]
        mbi, nnz, coef, i4 = to_product_layout(enc.mbs())
        fi = int(enc.frame_is_i())
        args = (mbi.ctypes.data, nnz.ctypes.data, coef.ctypes.data, w // 16, h // 16, h // 16, 0, fi)
        nb = hh.hh_cabac_bins(*args, None, 0, i4.ctypes.data)
        bins = np.zeros(nb, np.uint16)
        hh.hh_cabac_bins(*args, bins.ctypes.data, nb, i4.ctypes.data)
        bits = oracle.slice_header_bits(fi, t, 1)
        rbsp = oracle.cabac_code_bins(bins, fi, 20, int(bits, 2), len(bits))[0]
        assert len(nals) == 1 and nals[0][5:] == escape(rbsp), "frame %d" % t


def test_golden_bin_coder_rejects_malformed_bins(oracle):
    for bad in ([5], [5, BIN_TERM], [END, END], [NCTX, END], [BIN_BYPASS | BIN_TERM, END], [1 << 12, END]):
        with pytest.raises(ValueError):
            oracle.cabac_code_bins(np.array(bad, np.uint16), 1, 24)


def lps_flags(oracle, bins, frame_i, qp):
    pre = oracle.cabac_code_bins(bins, frame_i, qp)[1]
    regular = (bins & (BIN_BYPASS | BIN_TERM)) == 0
    return regular, regular & ((((bins >> 15) & 1) ^ (pre & 1)) == 1)


@pytest.mark.parametrize("family", FAMILIES)
def test_family_has_its_property(oracle, gen, family):
    n = LENGTHS[-1]
    bins = gen(family, n)
    assert bins[-1] == END and np.count_nonzero(bins == END) == 1
    regular, lps = lps_flags(oracle, bins, 1, 24)
    assert np.all((bins[regular] & 0x3ff) < NCTX)
    nreg, nlps = int(regular.sum()), int(lps.sum())
    ctx = bins[regular] & 0x3ff
    if family == "uniform":
        assert 0.08 < np.mean((bins & BIN_BYPASS) != 0) < 0.12
        assert 0.015 < np.mean(bins == BIN_TERM) < 0.025
        assert np.unique(ctx).size == NCTX
    if family in ("hot_mps", "hot_lps"):
        assert np.mean(ctx == HOT) >= 0.95
        assert np.all((bins[RES_TILE:2 * RES_TILE] & 0x3ff) == HOT) and np.all(regular[RES_TILE:2 * RES_TILE])
        # the hot context's bins per resolver tile leave every remainder mod 4 (the walk's one-to-three-bin tail)
        per_tile = [((bins[t:t + RES_TILE][regular[t:t + RES_TILE]] & 0x3ff) == HOT).sum() % 4 for t in range(0, n - RES_TILE, RES_TILE)]
        assert {1, 2, 3} <= set(per_tile)
        assert (nlps / nreg < 0.1) if family == "hot_mps" else (nlps / nreg > 0.5)
    if family == "mps_only":
        assert nlps == 0 and nreg > 0.8 * n
    if family == "sparse_lps":  # whole coder tiles without a chunk start; the look-ahead of a tile runs past 62 bins
        at = np.flatnonzero(lps)
        assert 4 <= nlps <= 8 and np.diff(at).min() > CP_TB
        assert set(range(n // CP_TB)) - set((at // CP_TB).tolist())
    if family == "lps_heavy":
        assert nlps / nreg > 0.8
        assert lps[CP_TB - 1] and lps[2 * CP_TB - 1]
        assert lps[np.flatnonzero(regular)[-1]]
    if family == "alternating":
        assert nlps / nreg > 0.3
    if family == "carry":
        _, _, (run, carry, _) = oracle.cabac_code_bins(bins, 1, 24)
        assert run >= 70000
    if family == "natural":
        assert np.unique(ctx).size > 100 and 0.02 < np.mean((bins & BIN_BYPASS) != 0) < 0.5


@pytest.mark.parametrize("run,carry", CARRY_RUNS)
def test_carry_sequences_reach_long_outstanding_runs(oracle, run, carry):
    """The golden coder reports the longest outstanding run and how it ended: both endings, at every length."""
    bins = np.append(carry_segment(run, carry), np.uint16(END))
    assert oracle.cabac_code_bins(bins, 1, 24)[2][:2] == (run, carry)


def build_gpu_harness(so=HARNESS_SO):
    deps = [HARNESS_SRC] + [os.path.join(CSRC, f) for f in ("kernels.cuh", "entropy.cuh", "h264_core.cuh", "h264_tables.h")]
    if os.path.exists(so) and all(os.path.getmtime(d) <= os.path.getmtime(so) for d in deps):
        return so
    fd, tmp = tempfile.mkstemp(suffix=".so", dir=os.path.dirname(so))
    os.close(fd)
    try:
        subprocess.check_call([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler",
                               "-fPIC", "-shared", "--cudart", "static", "-o", tmp, HARNESS_SRC])
        os.replace(tmp, so)
    finally:
        if os.path.exists(tmp):
            os.unlink(tmp)
    return so


def test_gpu_harness_cross_compiles_for_sm100a(tmp_path):
    if not os.path.exists(NVCC):
        pytest.skip("nvcc not installed")
    so = build_gpu_harness(str(tmp_path / "libcabac_gpu_harness.so"))
    out = subprocess.run(["nm", "-D", so], capture_output=True, text=True).stdout
    assert " T cg_cabac_backend" in out and " T cg_nal_assembly" in out


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the kernels
# ---------------------------------------------------------------------------------------------------------------------
SENTINEL = 0xDEADBEEF


@pytest.fixture(scope="module")
def cg():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    L = C.CDLL(build_gpu_harness())
    p, i, u, ull = C.c_void_p, C.c_int, C.c_uint, C.c_ulonglong
    L.cg_cabac_backend.argtypes = [p, ull] + [i] * 8 + [p] * 4 + [u, ull] + [p] * 4
    L.cg_nal_assembly.argtypes = [p, u, p, i, i, i, i, p, i, i, ull, p, p, p, p, p]
    return L


class Unit:
    def __init__(self, off, bins, frame_i, qp, k, oracle):
        self.off, self.bins = off, bins
        self.hdr = header(k)
        if bins.size:
            self.rbsp, self.pre, self.stats = oracle.cabac_code_bins(bins, frame_i, qp, *self.hdr)
        else:
            self.rbsp, self.pre, self.stats = b"", np.zeros(0, np.uint8), (0, 0, 0)


def run_backend(cg, pool, units, nslices, qp, gop_len=1, gop_pos0=0, step=None, rbsp_cap=None, limb_cap=None):
    """units: {u: Unit} (u = frame * nslices + slice); U = (max u // nslices + 1) * nslices units are addressed."""
    nframes = max(units) // nslices + 1
    U = nframes * nslices
    nlanes, frame0, stride, nfr = step or (nframes, 0, 1, nframes)
    if rbsp_cap is None:
        rbsp_cap = (max(len(x.rbsp) for x in units.values()) + 64 + 128 + 255) & ~255
    if limb_cap is None:
        limb_cap = rbsp_cap // 2 + 8
    off = np.zeros(U, np.uint64)
    ln = np.zeros(U, np.uint32)
    hb = np.zeros(U, np.uint64)
    hn = np.zeros(U, np.int32)
    for k, x in units.items():
        off[k], ln[k], hb[k], hn[k] = x.off, x.bins.size, x.hdr[0], x.hdr[1]
    pool_out = np.array(pool, np.uint16)
    rbsp = np.zeros(U * rbsp_cap, np.uint8)
    rlen = np.full(U, SENTINEL, np.uint32)
    hist = np.zeros(464, np.uint64)
    err = np.zeros(1, np.int32)
    r = cg.cg_cabac_backend(pool_out.ctypes.data, pool_out.size, nslices, qp, gop_len, gop_pos0, nlanes, frame0, stride,
                            nfr, off.ctypes.data, ln.ctypes.data, hb.ctypes.data, hn.ctypes.data, rbsp_cap, limb_cap,
                            rbsp.ctypes.data, rlen.ctypes.data, hist.ctypes.data, err.ctypes.data)
    assert r == 0, "harness: %d (%s)" % (r, "guard region of device buffer %d overwritten" % (-100 - r) if r <= -100 else "CUDA error")
    return pool_out, rbsp.reshape(U, rbsp_cap), rlen, hist, int(err[0])


def check_backend(cg, pool, units, nslices, qp, gop_len=1, gop_pos0=0, step=None, what=""):
    """Runs the back end and checks records, untouched pool bytes, RBSP, idle units, ctx_hist and the error word."""
    nframes = max(units) // nslices + 1
    nlanes, frame0, stride, nfr = step or (nframes, 0, 1, nframes)
    launched = {f * nslices + k for f in (frame0 + l * stride for l in range(nlanes)) if f < nfr for k in range(nslices)}
    pool_out, rbsp, rlen, hist, err = run_backend(cg, pool, units, nslices, qp, gop_len, gop_pos0, step)
    assert err == 0, what
    touched = np.zeros(pool.size, bool)
    want_hist = np.zeros(464, np.int64)
    for u, x in sorted(units.items()):
        n = x.bins.size
        if u not in launched:
            assert rlen[u] == SENTINEL and np.all(rbsp[u] == 0xcd), "%s unit %d is not coded" % (what, u)
            continue
        if n == 0:
            assert rlen[u] == 0, "%s unit %d has no bins" % (what, u)
            continue
        touched[x.off:x.off + n] = True
        got, want = pool_out[x.off:x.off + n], records(x.bins, x.pre)
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, "%s unit %d: record of bin %d is %#x, want %#x (bin %#x)" % (
            what, u, bad[0], got[bad[0]], want[bad[0]], x.bins[bad[0]])
        assert rlen[u] == len(x.rbsp), "%s unit %d: rbsp_len %d, want %d" % (what, u, rlen[u], len(x.rbsp))
        g = rbsp[u, :len(x.rbsp)].tobytes()
        if g != x.rbsp:
            first = next(i for i in range(len(g)) if g[i] != x.rbsp[i])
            pytest.fail("%s unit %d: RBSP byte %d of %d differs" % (what, u, first, len(g)))
        regular = (x.bins & (BIN_BYPASS | BIN_TERM)) == 0
        want_hist += np.bincount(x.bins[regular] & 0x3ff, minlength=464)
    assert np.array_equal(pool_out[~touched], pool[~touched]), "%s: pool bytes outside the slices changed" % what
    assert np.array_equal(hist.astype(np.int64), want_hist), what


def junk_pool(size, seed):
    return np.random.default_rng(seed).integers(0, 1 << 16, size, dtype=np.uint16)


@pytest.mark.gpu
@pytest.mark.parametrize("n", LENGTHS)
@pytest.mark.parametrize("family", FAMILIES)
def test_backend_matches_golden_coder(oracle, cg, gen, family, n):
    frame_i, qp = case_params(n)
    bins = gen(family, n, frame_i, qp)
    off = 16 + n % 8
    pool = junk_pool(off + n + 40, n)
    pool[off:off + n] = bins
    check_backend(cg, pool, {0: Unit(off, bins, frame_i, qp, n, oracle)}, 1, qp, gop_len=1 if frame_i else 2,
                  gop_pos0=0 if frame_i else 1, what="%s n=%d" % (family, n))


@pytest.mark.gpu
@pytest.mark.parametrize("mis", range(8))
def test_backend_slice_at_every_pool_alignment(oracle, cg, gen, mis):
    """The slice's first bin at every element offset inside a 16-byte vector; lengths end at every offset too."""
    for family, n in (("uniform", 9000 + 3 * mis), ("hot_lps", 4096 + 2 * mis + 1), ("natural", 31745 - mis)):
        bins = gen(family, n)
        off = 64 + mis
        pool = junk_pool(off + n + 64, mis)
        pool[off:off + n] = bins
        check_backend(cg, pool, {0: Unit(off, bins, 1, 24, mis, oracle)}, 1, 24, what="%s mis=%d" % (family, mis))


@pytest.mark.gpu
@pytest.mark.parametrize("nslices", [3, 17])
def test_backend_slices_back_to_back(oracle, cg, gen, nslices):
    """Slices of one picture lie back to back from an odd start; one slice has no bins."""
    rng = np.random.default_rng(nslices)
    lens = [int(v) for v in rng.integers(1, 24000, nslices)]
    lens[1] = 0
    lens[-1] = 4097
    off, pieces, units = 5, [], {}
    for k, n in enumerate(lens):
        bins = gen(FAMILIES[k % len(FAMILIES)], n) if n else np.zeros(0, np.uint16)
        units[k] = Unit(off, bins, 1, 24, k, oracle)
        pieces.append(bins)
        off += n
    pool = junk_pool(off + 11, nslices)
    pool[5:off] = np.concatenate(pieces)
    check_backend(cg, pool, units, nslices, 24, what="%d slices" % nslices)


@pytest.mark.gpu
def test_backend_lanes_idle_lane_and_mixed_picture_types(oracle, cg, gen):
    """Three lanes hold frames 1, 3 and 5 of a five-frame clip (the third lane idles); gop_pos0 makes frame 1 an I
    frame and frame 3 a P frame.  The units of frames no lane holds must stay untouched."""
    nslices, qp, gop_len, gop_pos0 = 2, 30, 3, 2
    step = (3, 1, 2, 5)
    units, off, pieces = {}, 8, []
    for f in range(5):
        frame_i = int((gop_pos0 + f) % gop_len == 0)
        for k in range(nslices):
            u = f * nslices + k
            bins = gen(("uniform", "natural", "hot_mps", "carry")[u % 4], 5000 + 997 * u, frame_i, qp)
            units[u] = Unit(off, bins, frame_i, qp, u, oracle)
            pieces.append(bins)
            off += bins.size
    pool = junk_pool(off + 8, 3)
    pool[8:off] = np.concatenate(pieces)
    check_backend(cg, pool, units, nslices, qp, gop_len, gop_pos0, step, what="lanes")


@pytest.mark.gpu
@pytest.mark.parametrize("qp", [1, 24, 47])
@pytest.mark.parametrize("frame_i", [1, 0])
def test_backend_every_qp_and_picture_type(oracle, cg, gen, qp, frame_i):
    units, off, pieces = {}, 0, []
    for k, (family, n) in enumerate((("uniform", 40000), ("hot_mps", 20000), ("mps_only", 33000), ("lps_heavy", 31807))):
        bins = gen(family, n, frame_i, qp)
        units[k] = Unit(off, bins, frame_i, qp, k, oracle)
        pieces.append(bins)
        off += bins.size
    check_backend(cg, np.concatenate(pieces), units, 4, qp, gop_len=1 if frame_i else 2, gop_pos0=0 if frame_i else 1,
                  what="qp %d %s" % (qp, "I" if frame_i else "P"))


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["limb_cap", "rbsp_cap"])
def test_backend_capacity_overflow_is_error_3(oracle, cg, which):
    """Caps just large enough for a 70 000-bit carry run code it exactly; one limb (or byte) less is error 3 with
    rbsp_len 0, and every write stays inside the buffers."""
    bins = np.concatenate([carry_segment(70000, 1), carry_segment(9000, 0), np.array([END], np.uint16)])
    unit = Unit(0, bins, 1, 24, 3, oracle)
    t_end = unit.stats[2] - 2  # the coder's last stream bit position; the stop bit follows it
    need_limbs = ((t_end + 8) >> 4) + 2
    need_rbsp = len(unit.rbsp) + 64
    roomy_rbsp = need_rbsp + 4096
    for cap_r, cap_l, ok in ((need_rbsp, need_limbs, True),
                             (roomy_rbsp, need_limbs - 1, False) if which == "limb_cap" else (need_rbsp - 1, need_limbs + 64, False)):
        pool_out, rbsp, rlen, _, err = run_backend(cg, bins, {0: unit}, 1, 24, rbsp_cap=cap_r, limb_cap=cap_l)
        if ok:
            assert err == 0 and rlen[0] == len(unit.rbsp) and rbsp[0, :rlen[0]].tobytes() == unit.rbsp
        else:
            assert err == 3 and rlen[0] == 0, (which, err, rlen[0])
        assert np.array_equal(pool_out, records(bins, unit.pre))


# ---------------------------------------------------------------------------------------------------------------------
# GPU: NAL assembly
# ---------------------------------------------------------------------------------------------------------------------
def escape(rbsp):
    """Sequential emulation prevention (7.4.1): after 00 00, a byte <= 3 gets an 0x03 in front."""
    out, zeros = bytearray(), 0
    for b in rbsp:
        if zeros >= 2 and b <= 3:
            out.append(3)
            zeros = 0
        out.append(b)
        zeros = zeros + 1 if b == 0 else 0
    return bytes(out)


def pack(units, nslices, gop_len, first_frame_index, ps, mode):
    """Python packer: [SPS + PPS] start code, NAL header (IDR 0x65, P 0x41), escaped RBSP per unit."""
    out, offs, fbytes = bytearray(), [], [0] * (len(units) // nslices)
    for u, r in enumerate(units):
        offs.append(len(out))
        fr = u // nslices
        first = u % nslices == 0
        idr = (first_frame_index + fr) % gop_len == 0
        nal = bytearray()
        if first and ((mode == 1 and u == 0) or (mode == 2 and idr)):
            nal += ps
        nal += b"\0\0\0\1" + bytes([0x65 if idr else 0x41]) + escape(r)
        out += nal
        fbytes[fr] += len(nal)
    return bytes(out), offs, fbytes


def rbsp_unit(rng, n):
    """n RBSP bytes from {0, 0, 0, 1, 2, 3, 4, 255}, zero runs ending at the 64-byte chunk edges, a 00 00 03, and a
    last byte that is not 0 (as the coder's stop bit guarantees)."""
    b = rng.choice(np.array([0, 0, 0, 1, 2, 3, 4, 255], np.uint8), size=n)
    for end in (int(rng.integers(62, 67)), int(rng.integers(126, 131))):
        run = int(rng.integers(1, 201))
        if end < n:
            b[max(0, end - run):end] = 0
            b[end] = rng.integers(0, 4)
    if n > 40:
        b[30:33] = (0, 0, 3)
    b[-1] = rng.choice(np.array([1, 2, 3, 4, 255], np.uint8))
    return b


def run_nal(cg, units, rbsp_cap, nslices, gop_len, ffi, ps, mode, out_cap, out_init=None):
    U = len(units)
    rb = np.zeros((U, rbsp_cap), np.uint8)
    rl = np.zeros(U, np.uint32)
    for u, r in enumerate(units):
        rb[u, :len(r)] = np.frombuffer(r, np.uint8)
        rl[u] = len(r)
    out = np.full(out_cap, 0x5a, np.uint8) if out_init is None else out_init.copy()
    nal_off = np.zeros(U, np.uint64)
    fb = np.zeros(U // nslices, np.int32)
    total = np.zeros(1, np.uint64)
    err = np.zeros(1, np.int32)
    psb = np.frombuffer(ps.ljust(64, b"\0"), np.uint8).copy()
    r = cg.cg_nal_assembly(rb.ctypes.data, rbsp_cap, rl.ctypes.data, U, nslices, gop_len, ffi, psb.ctypes.data, len(ps),
                           mode, out_cap, out.ctypes.data, nal_off.ctypes.data, fb.ctypes.data, total.ctypes.data,
                           err.ctypes.data)
    assert r == 0, "harness: %d" % r
    return out, nal_off, fb, int(total[0]), int(err[0])


PS = bytes([0, 0, 0, 1, 0x67, 0x4d, 0x40, 0x29, 0xab, 0, 0, 0, 1, 0x68, 0xee, 0x3c, 0x80])
NAL_LENS = [1, 2, 3, 4, 5, 63, 64, 65, 127, 128, 129]


@pytest.mark.gpu
@pytest.mark.parametrize("ffi", [0, 5])
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("nunits,nslices", [(1, 1), (3, 1), (1025, 1), (2100, 1), (4, 4), (12, 4), (1028, 4), (2100, 4)])
def test_nal_assembly_matches_python_packer(cg, nunits, nslices, mode, ffi):
    rng = np.random.default_rng([nunits, nslices, mode, ffi])
    big = nunits <= 12  # a unit of 70 000 bytes (over 1 024 chunks) where the unit count keeps the buffers small
    rbsp_cap = 70016 if big else 16448  # both above 16 KB: more than 256 chunks, more than one block per unit
    lens = [NAL_LENS[u % len(NAL_LENS)] if u % 61 else int(rng.integers(130, 16400)) for u in range(nunits)]
    if big:
        lens[nunits // 2] = 70000
    units = [rbsp_unit(rng, n).tobytes() for n in lens]
    want, offs, fbytes = pack(units, nslices, 3, ffi, PS, mode)
    out, nal_off, fb, total, err = run_nal(cg, units, rbsp_cap, nslices, 3, ffi, PS, mode, len(want) + 100)
    assert err == 0 and total == len(want)
    assert out[:total].tobytes() == want
    assert np.all(out[total:] == 0x5a)
    assert nal_off.tolist() == offs and fb.tolist() == fbytes


@pytest.mark.gpu
def test_nal_assembly_out_cap_overflow_is_error_4(cg):
    rng = np.random.default_rng(9)
    units = [rbsp_unit(rng, n).tobytes() for n in (700, 65, 3000, 129)]
    want = pack(units, 2, 3, 0, PS, 1)[0]
    out, _, _, total, err = run_nal(cg, units, 4096, 2, 3, 0, PS, 1, len(want))
    assert err == 0 and total == len(want) and out.tobytes() == want
    init = np.random.default_rng(1).integers(0, 256, len(want) - 1, dtype=np.uint8)
    out, _, _, total, err = run_nal(cg, units, 4096, 2, 3, 0, PS, 1, len(want) - 1, init)
    assert err == 4 and total == 0
    assert np.array_equal(out, init), "nothing is written when the stream does not fit"


@pytest.mark.gpu
def test_bins_to_packed_stream(oracle, cg, gen):
    """Bins -> back end -> NAL assembly equals the Python packing of the golden coder's RBSP (3 slices, I then P)."""
    nslices, qp, gop_len = 3, 24, 2
    units, off, pieces = {}, 0, []
    for u in range(2 * nslices):
        frame_i = int(u < nslices)
        bins = gen(("natural", "carry", "uniform")[u % 3], 20000 + 4099 * u, frame_i, qp)
        units[u] = Unit(off, bins, frame_i, qp, u, oracle)
        pieces.append(bins)
        off += bins.size
    _, rbsp, rlen, _, err = run_backend(cg, np.concatenate(pieces), units, nslices, qp, gop_len)
    assert err == 0
    got_units = [rbsp[u, :rlen[u]].tobytes() for u in range(2 * nslices)]
    want = pack([units[u].rbsp for u in range(2 * nslices)], nslices, gop_len, 0, PS, 1)[0]
    out, _, _, total, err = run_nal(cg, got_units, rbsp.shape[1], nslices, gop_len, 0, PS, 1, len(want) + 64)
    assert err == 0 and out[:total].tobytes() == want
