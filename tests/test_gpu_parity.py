"""Parity tests proper (run on the B200 box: pytest -m gpu).  Everything goes through the C ABI
(include/cedar_b200.h via ctypes).  Bar: bit-exact -- bytestream, every intermediate (macroblock
records, levels, reconstruction before and after deblocking) and the luma SSE equal the CPU golden
model's on the same seeded inputs; at BASELINE.json's full sizes, size-independent properties:
an independent decoder reproduces the encoder's reconstruction, and the GOP-parallel clip path
equals the frame-at-a-time path and is independent of the number of GOPs in flight."""
import numpy as np
import pytest
import torch

import avdec
from common import content, make_clip, oracle_encode_clip, split_frame

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():
    pytest.skip("no CUDA device", allow_module_level=True)

import cedarx_h264_encoder_b200 as cx  # noqa: E402
from cedarx_h264_encoder_b200 import api, synth  # noqa: E402


def test_library_is_loaded_and_launches_kernels(product_lib):
    with cx.Encoder(api.make_config(64, 48)) as enc:
        y, c = content("synth", 64, 48, 0)
        assert len(enc.encode(y, c)) > 0
        assert enc.launch_count() >= 10


@pytest.mark.parametrize("cabac", [0, 1])
@pytest.mark.parametrize("kind,qp,me", [("synth", 24, 8), ("noise", 30, 8), ("static", 30, 8), ("shift", 24, 16),
                                        ("noise", 1, 8), ("synth", 47, 8), ("flat", 12, 8)])
def test_frame_mode_every_stage_matches_oracle(oracle, kind, qp, me, cabac):
    w, h, gop, n = 96, 80, 3, 5
    gold = oracle.Encoder(oracle.make_config(w, h, qp=qp, gop=gop, cabac=cabac, me_range=me))
    with cx.Encoder(api.make_config(w, h, qp=qp, gop=gop, cabac=cabac, me_range=me)) as enc:
        for t in range(n):
            y, c = content(kind, w, h, t)
            want, got = gold.encode(y, c), enc.encode(y, c)
            for p, (a, b) in enumerate(zip(gold.source(), enc.debug_planes(0))):
                assert np.array_equal(a, b), "ingest plane %d frame %d" % (p, t)
            mbs = gold.mbs()
            mbi, nnz, coef = enc.debug_syntax()
            for k in ("type", "i16_mode", "chroma_mode", "cbp", "mv", "mvd"):
                assert np.array_equal(mbs[k], mbi[k]), "mb.%s frame %d" % (k, t)
            assert np.array_equal(mbs["nnz"], nnz[:, :27]), "nnz frame %d" % t
            assert np.array_equal(mbs["coef"], coef), "levels frame %d" % t
            for p, (a, b) in enumerate(zip(gold.recon_unfiltered(), enc.debug_planes(1))):
                assert np.array_equal(a, b), "recon before deblocking plane %d frame %d" % (p, t)
            for p, (a, b) in enumerate(zip(gold.recon(), enc.debug_planes(2))):
                assert np.array_equal(a, b), "recon after deblocking plane %d frame %d" % (p, t)
            assert got == want, "bytestream frame %d" % t
            assert gold.sse_y() == enc.sse_y(1)[0]
    gold.close()


@pytest.mark.parametrize("w,h,fmt,me", [(854, 480, 0, 16), (86, 50, 0, 8), (64, 48, 1, 8), (16, 16, 0, 8), (32, 16, 0, 4),
                                        (16, 64, 0, 16), (176, 144, 0, 16), (352, 288, 0, 32)])
def test_frame_mode_shapes_and_formats(oracle, w, h, fmt, me):
    """ragged sizes (edge replication), NV16 ingest, single-macroblock pictures, other search ranges"""
    gold = oracle.Encoder(oracle.make_config(w, h, qp=25, gop=25, cabac=1, fmt=fmt, me_range=me))
    with cx.Encoder(api.make_config(w, h, qp=25, gop=25, cabac=1, fmt=fmt, me_range=me)) as enc:
        for t in range(3):
            y, c = content("synth", w, h, t, fmt)
            assert enc.encode(y, c) == gold.encode(y, c), "frame %d" % t
    gold.close()


@pytest.mark.parametrize("me", [64, 1, 2, 3, 20, 32, 33, 47])
def test_me_ranges(oracle, me):
    """Every search-tile geometry of me_kernel: 4 x 4 macroblocks up to R = 32 (compiled-in row stride at 16, generic
    otherwise), 2 x 1 above (R = 33 shares the row stride of R = 16, R = 64 has its own instantiation), and the ranges
    with fewer than four row offsets per column."""
    w, h = 208, 160
    gold = oracle.Encoder(oracle.make_config(w, h, qp=25, gop=25, cabac=0, me_range=me))
    with cx.Encoder(api.make_config(w, h, qp=25, gop=25, cabac=0, me_range=me)) as enc:
        for t in range(2):
            y, c = content("shift", w, h, 3 * t)
            assert enc.encode(y, c) == gold.encode(y, c)
            assert np.array_equal(gold.mbs()["mv"], enc.debug_syntax()[0]["mv"])
    gold.close()


@pytest.mark.parametrize("first,second", [(20, 8), (16, 33), (63, 64)])
def test_me_ranges_of_two_live_handles(oracle, first, second):
    """Two handles on one device whose ranges share an me_kernel instantiation (generic, 27-word and 43-word row
    stride), the second needing less shared memory: its open() must not take from the first what the first's launches
    need.  I and P frame through the first, the second, the first again."""
    w, h = 208, 160
    golds = [oracle.Encoder(oracle.make_config(w, h, qp=25, gop=25, cabac=0, me_range=me)) for me in (first, second)]
    with cx.Encoder(api.make_config(w, h, qp=25, gop=25, cabac=0, me_range=first)) as a, \
            cx.Encoder(api.make_config(w, h, qp=25, gop=25, cabac=0, me_range=second)) as b:
        for i, enc in ((0, a), (1, b), (0, a)):
            for t in range(2):
                y, c = content("shift", w, h, 3 * t)
                assert enc.encode(y, c) == golds[i].encode(y, c), "handle %d frame %d" % (i, t)
                assert np.array_equal(golds[i].mbs()["mv"], enc.debug_syntax()[0]["mv"]), "handle %d frame %d" % (i, t)
    for g in golds:
        g.close()


@pytest.mark.parametrize("cabac", [0, 1])
@pytest.mark.parametrize("lanes", [0, 1, 3])
def test_clip_mode_matches_oracle(oracle, cabac, lanes):
    w, h, n, gop = 96, 80, 14, 4
    clip = make_clip("synth", w, h, n)
    want, sizes, _ = oracle_encode_clip(clip, w, h, qp=24, gop=gop, cabac=cabac, me_range=8)
    with cx.Encoder(api.make_config(w, h, qp=24, gop=gop, cabac=cabac, me_range=8, max_clip_frames=n,
                                    gops_in_flight=lanes)) as enc:
        got, gsz = enc.encode_clip(clip)
        assert got == want and gsz.tolist() == sizes
        got2, _ = enc.encode_clip(clip)  # the handle is reusable and deterministic
        assert got2 == want


@pytest.mark.parametrize("lanes", [0, 2])
def test_paced_upload_matches_oracle(oracle, lanes):
    """The copies of pass j + 1 are issued behind the ingest of pass j (encoder.cu upload_pass).  Different clips back
    to back through one handle (a stale frame would show), several waves of GOPs, a short last GOP, a clip shorter than
    the one before, and an upload that covers more frames than the encode."""
    w, h, n, gop = 96, 80, 14, 4
    clips = [make_clip(kind, w, h, m) for kind, m in (("synth", n), ("noise", n), ("shift", 9), ("static", n))]
    want = [oracle_encode_clip(c, w, h, qp=27, gop=gop, cabac=1, me_range=8)[0] for c in clips]
    with cx.Encoder(api.make_config(w, h, qp=27, gop=gop, cabac=1, me_range=8, max_clip_frames=n,
                                    gops_in_flight=lanes)) as enc:
        for _ in range(2):
            for c, wnt in zip(clips, want):
                assert enc.encode_clip(c)[0] == wnt
        # upload 14 frames, encode the first 8 and then all 14 without another upload
        enc.clip_input(n)[:] = clips[1].reshape(n, -1)
        enc.clip_upload(n)
        enc.clip_encode(8, 0)
        enc.clip_download(8)
        enc.clip_encode(n, 0)
        assert enc.clip_download(n)[0].tobytes() == want[1]


def test_handles_on_their_own_threads_do_not_interfere(oracle):
    """bench.py and INTEGRATION.md section 4 drive two or three handles per GPU, each from its own host thread: handles
    share nothing, so every one of them must still produce the oracle's bytes (different content, entropy coder and
    slice layout and QP per handle, several rounds, all in flight together)."""
    import threading
    w, h, n, gop = 96, 80, 13, 4
    jobs = [("synth", 1, 0, 27), ("static", 0, 0, 30), ("synth", 1, 2, 22)]
    want, encs, clips = [], [], []
    for kind, cabac, rows, qp in jobs:
        clip = make_clip(kind, w, h, n)
        want.append(oracle_encode_clip(clip, w, h, qp=qp, gop=gop, cabac=cabac, me_range=8, slice_rows=rows)[0])
        clips.append(clip)
        encs.append(cx.Encoder(api.make_config(w, h, qp=qp, gop=gop, cabac=cabac, me_range=8, max_clip_frames=n,
                                               gops_in_flight=2, slice_rows=rows)))
    got = [[] for _ in jobs]

    def work(i):
        for _ in range(6):
            got[i].append(encs[i].encode_clip(clips[i])[0])
    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(jobs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for e in encs:
        e.close()
    for i in range(len(jobs)):
        assert len(got[i]) == 6 and all(g == want[i] for g in got[i]), jobs[i]


def test_clip_mode_later_gops_carry_no_parameter_sets(oracle):
    """first_frame_index != 0: a rank that owns later GOPs emits no SPS/PPS (cedar.c:1058-1061), so
    rank streams concatenate to the single stream."""
    w, h, n, gop = 64, 48, 9, 3
    clip = make_clip("synth", w, h, n)
    want, sizes, _ = oracle_encode_clip(clip, w, h, qp=26, gop=gop, cabac=1, me_range=8)
    with cx.Encoder(api.make_config(w, h, qp=26, gop=gop, cabac=1, me_range=8, max_clip_frames=n)) as enc:
        a, _ = enc.encode_clip(clip[:3], first_frame_index=0)
        b, _ = enc.encode_clip(clip[3:], first_frame_index=3)
        assert a + b == want
        with pytest.raises(OSError):
            enc.encode_clip(clip[1:4], first_frame_index=1)  # clips start at a GOP boundary


def test_overflow_is_reported_not_silent(monkeypatch):
    monkeypatch.setenv("CEDAR_B200_BINS_PER_MB", "8")
    monkeypatch.setenv("CEDAR_B200_NO_GROW", "1")
    clip = make_clip("noise", 64, 48, 2)
    with cx.Encoder(api.make_config(64, 48, qp=10, gop=25, cabac=1, me_range=8, max_clip_frames=2)) as enc:
        with pytest.raises(OSError):
            enc.encode_clip(clip)


@pytest.mark.parametrize("cabac", [0, 1])
def test_clip_that_overflows_the_heuristic_bounds_is_encoded_again_with_larger_buffers(oracle, monkeypatch, cabac):
    """The entropy buffers of clip mode are sized by a per-macroblock heuristic.  Noise at a low QP exceeds it: the
    library enlarges the buffers and encodes the resident clip again; the caller sees the oracle's bytes, not an error."""
    if cabac:
        monkeypatch.setenv("CEDAR_B200_BINS_PER_MB", "64")
    w, h, n, gop = 96, 80, 9, 4
    clip = make_clip("noise", w, h, n)
    want, sizes, _ = oracle_encode_clip(clip, w, h, qp=21, gop=gop, cabac=cabac, me_range=8)
    with cx.Encoder(api.make_config(w, h, qp=21, gop=gop, cabac=cabac, me_range=8, max_clip_frames=n)) as enc:
        got, gsz = enc.encode_clip(clip)
        assert got == want and gsz.tolist() == sizes
        got2, _ = enc.encode_clip(clip)  # the enlarged buffers stay
        assert got2 == want


@pytest.mark.parametrize("name,w,h,fmt,gop,n,me", [("720p", 1280, 720, 0, 30, 31, 16), ("1080p", 1920, 1088, 0, 60, 61, 16),
                                                   ("1080p-nv16", 1920, 1088, 1, 60, 3, 16),
                                                   ("2160p-me64", 3840, 2160, 0, 60, 3, 64)])
def test_full_size_properties(name, w, h, fmt, gop, n, me):
    """BASELINE.json shapes: (1) clip path == frame-at-a-time path, (2) independent of GOPs in flight,
    (3) libavcodec decodes the stream to exactly the encoder's reconstruction (last frame of each path),
    (4) Y-PSNR is sane."""
    clip = synth.synth_clip(w, h, list(range(n)), fmt).numpy()
    with cx.Encoder(api.make_config(w, h, qp=25, gop=gop, cabac=1, fmt=fmt, me_range=me, max_clip_frames=n, gops_in_flight=2)) as enc:
        stream, sizes = enc.encode_clip(clip)
        sse = enc.sse_y(n)
    with cx.Encoder(api.make_config(w, h, qp=25, gop=gop, cabac=1, fmt=fmt, me_range=me, max_clip_frames=n, gops_in_flight=1)) as enc:
        stream1, _ = enc.encode_clip(clip)
    assert stream == stream1, "result depends on the number of GOPs in flight"
    with cx.Encoder(api.make_config(w, h, qp=25, gop=gop, cabac=1, fmt=fmt, me_range=me)) as enc:
        frames = b""
        for t in range(n):
            frames += enc.encode(*split_frame(clip[t], w, h, fmt))
        last_recon = enc.debug_planes(2)
    assert frames == stream, "clip path differs from the frame-at-a-time path"
    dec = avdec.decode(stream)
    assert len(dec) == n
    W16, H16 = (w + 15) // 16 * 16, (h + 15) // 16 * 16
    for p in range(3):
        assert np.array_equal(dec[-1][p], last_recon[p]), "decoder != encoder reconstruction (plane %d)" % p
    # SSE reported by the encoder == SSE of the decoded picture against the (padded) input
    y_in = np.pad(split_frame(clip[-1], w, h, fmt)[0], ((0, H16 - h), (0, W16 - w)), mode="edge").astype(np.int64)
    assert int(((dec[-1][0].astype(np.int64) - y_in) ** 2).sum()) == int(sse[-1])
    psnr = 10 * np.log10(255.0 ** 2 / (sse.sum() / (n * W16 * H16)))
    assert psnr > 34.0, psnr


def _assert_every_stage_equal(gold, enc, t):
    for p, (a, b) in enumerate(zip(gold.source(), enc.debug_planes(0))):
        assert np.array_equal(a, b), "ingest plane %d frame %d" % (p, t)
    mbs = gold.mbs()
    mbi, nnz, coef = enc.debug_syntax()
    for k in ("type", "i16_mode", "chroma_mode", "cbp", "mv", "mvd"):
        assert np.array_equal(mbs[k], mbi[k]), "mb.%s frame %d" % (k, t)
    assert np.array_equal(mbs["nnz"], nnz[:, :27]), "nnz frame %d" % t
    assert np.array_equal(mbs["coef"], coef), "levels frame %d" % t
    for p, (a, b) in enumerate(zip(gold.recon_unfiltered(), enc.debug_planes(1))):
        assert np.array_equal(a, b), "recon before deblocking plane %d frame %d" % (p, t)
    for p, (a, b) in enumerate(zip(gold.recon(), enc.debug_planes(2))):
        assert np.array_equal(a, b), "recon after deblocking plane %d frame %d" % (p, t)
    assert gold.sse_y() == enc.sse_y(1)[0]


@pytest.mark.parametrize("name,w,h,fmt,n,me", [("720p", 1280, 720, 0, 3, 16), ("1080p", 1920, 1088, 0, 3, 16),
                                               ("1080p-nv16", 1920, 1088, 1, 3, 16), ("2160p-me64", 3840, 2160, 0, 2, 64)])
def test_full_size_every_stage_matches_oracle(oracle, name, w, h, fmt, n, me):
    """BASELINE.json's shapes against the golden model itself (not only against properties): motion vectors, levels,
    reconstruction before and after deblocking, SSE and bytes of 1 I + (n - 1) P frames, at the search geometry the
    benchmark runs (4 x 4 macroblock tiles with the compiled-in row stride at R = 16, 2 x 1 tiles at R = 64)."""
    gold = oracle.Encoder(oracle.make_config(w, h, qp=25, gop=60, cabac=1, fmt=fmt, me_range=me))
    with cx.Encoder(api.make_config(w, h, qp=25, gop=60, cabac=1, fmt=fmt, me_range=me)) as enc:
        for t in range(n):
            y, c = content("synth", w, h, t, fmt)
            want, got = gold.encode(y, c), enc.encode(y, c)
            _assert_every_stage_equal(gold, enc, t)
            assert got == want, "bytestream frame %d" % t
    gold.close()


@pytest.mark.parametrize("cabac", [1, 0])
def test_1080p_clip_mode_ten_gops_in_flight_matches_oracle(oracle, cabac):
    """The benchmark's geometry -- 1920x1088, ten closed GOPs in lock step -- against the golden model, byte for byte:
    30 frames as 10 GOPs of 1 I + 2 P, and the per-frame sizes."""
    w, h, gop, n = 1920, 1088, 3, 30
    clip = synth.synth_clip(w, h, list(range(n)), 0).numpy()
    want, sizes, _ = oracle_encode_clip(clip, w, h, qp=25, gop=gop, cabac=cabac, me_range=16)
    with cx.Encoder(api.make_config(w, h, qp=25, gop=gop, cabac=cabac, me_range=16, max_clip_frames=n,
                                    gops_in_flight=10)) as enc:
        got, gsz = enc.encode_clip(clip)
    assert gsz.tolist() == sizes
    assert got == want


def test_gpu_stream_decodes_bit_exactly_small(oracle):
    w, h, n = 176, 144, 6
    clip = make_clip("synth", w, h, n)
    _, _, recs = oracle_encode_clip(clip, w, h, keep_recon=True, qp=24, gop=3, cabac=1, me_range=16)
    with cx.Encoder(api.make_config(w, h, qp=24, gop=3, cabac=1, max_clip_frames=n)) as enc:
        stream, _ = enc.encode_clip(clip)
    dec = avdec.decode(stream)
    for r, d in zip(recs, dec):
        for p in range(3):
            assert np.array_equal(r[p], d[p])


# ---- slice_rows extension (north star: "MB rows per slice configurable, bitrate cost reported") ----------------
@pytest.mark.parametrize("cabac", [0, 1])
@pytest.mark.parametrize("kind,qp,rows", [("synth", 24, 1), ("noise", 30, 2), ("static", 30, 3), ("shift", 24, 2), ("noise", 1, 4)])
def test_slices_every_stage_matches_oracle(oracle, kind, qp, rows, cabac):
    w, h, gop, n = 96, 80, 3, 5
    gold = oracle.Encoder(oracle.make_config(w, h, qp=qp, gop=gop, cabac=cabac, me_range=8, slice_rows=rows))
    with cx.Encoder(api.make_config(w, h, qp=qp, gop=gop, cabac=cabac, me_range=8, slice_rows=rows)) as enc:
        for t in range(n):
            y, c = content(kind, w, h, t)
            want, got = gold.encode(y, c), enc.encode(y, c)
            mbs = gold.mbs()
            mbi, nnz, coef = enc.debug_syntax()
            for k in ("type", "i16_mode", "chroma_mode", "cbp", "mv", "mvd"):
                assert np.array_equal(mbs[k], mbi[k]), "mb.%s frame %d" % (k, t)
            assert np.array_equal(mbs["coef"], coef), "levels frame %d" % t
            for p, (a, b) in enumerate(zip(gold.recon(), enc.debug_planes(2))):
                assert np.array_equal(a, b), "recon after deblocking plane %d frame %d" % (p, t)
            assert got == want, "bytestream frame %d" % t
    gold.close()


@pytest.mark.parametrize("cabac", [0, 1])
@pytest.mark.parametrize("rows,lanes", [(1, 0), (2, 3), (4, 1), (5, 2)])
def test_slices_clip_mode_matches_oracle(oracle, rows, lanes, cabac):
    w, h, n, gop = 96, 80, 11, 4
    clip = make_clip("synth", w, h, n)
    want, sizes, _ = oracle_encode_clip(clip, w, h, qp=24, gop=gop, cabac=cabac, me_range=8, slice_rows=rows)
    with cx.Encoder(api.make_config(w, h, qp=24, gop=gop, cabac=cabac, me_range=8, max_clip_frames=n,
                                    gops_in_flight=lanes, slice_rows=rows)) as enc:
        got, gsz = enc.encode_clip(clip)
        assert got == want and gsz.tolist() == sizes


@pytest.mark.parametrize("cabac", [0, 1])
def test_slices_full_size_decode_and_bitrate_cost(cabac):
    """1080p, 4 rows per slice (17 slices): the independent decoder reproduces the encoder's reconstruction, the
    frame-at-a-time path equals the clip path, and the extra bits over one slice per picture stay moderate."""
    w, h, n, gop = 1920, 1088, 4, 60
    clip = synth.synth_clip(w, h, list(range(n)), 0).numpy()
    total = {}
    for rows in (0, 4):
        with cx.Encoder(api.make_config(w, h, qp=25, gop=gop, cabac=cabac, max_clip_frames=n, slice_rows=rows)) as enc:
            stream, sizes = enc.encode_clip(clip)
        total[rows] = len(stream)
        if rows:
            with cx.Encoder(api.make_config(w, h, qp=25, gop=gop, cabac=cabac, slice_rows=rows)) as enc:
                frames = b""
                for t in range(n):
                    frames += enc.encode(*split_frame(clip[t], w, h, 0))
                last_recon = enc.debug_planes(2)
            assert frames == stream
            dec = avdec.decode(stream)
            assert len(dec) == n
            for p in range(3):
                assert np.array_equal(dec[-1][p], last_recon[p])
    assert total[0] < total[4] < 1.10 * total[0], total


def test_sps_crop_and_auto_level_stream_matches_oracle(oracle):
    w, h = 100, 50
    gold = oracle.Encoder(oracle.make_config(w, h, qp=25, gop=2, cabac=1, me_range=8, sps_crop=1, auto_level=1))
    with cx.Encoder(api.make_config(w, h, qp=25, gop=2, cabac=1, me_range=8, sps_crop=1, auto_level=1)) as enc:
        stream = b""
        for t in range(3):
            y, c = content("synth", w, h, t)
            got = enc.encode(y, c)
            assert got == gold.encode(y, c), "frame %d" % t
            stream += got
    gold.close()
    dec = avdec.decode(stream)
    assert len(dec) == 3 and dec[0][0].shape == (h, w)


@pytest.mark.parametrize("rows", [0, 2])
def test_repeat_headers_makes_every_gop_decodable_on_its_own(oracle, rows):
    """repeat_headers: SPS + PPS before every IDR (frame mode == clip mode == oracle); a later GOP, cut out of the
    stream, decodes by itself -- what a rank of a GOP-parallel encode produces with first_frame_index != 0."""
    w, h, n, gop = 96, 80, 9, 3
    clip = make_clip("synth", w, h, n)
    want, sizes, recs = oracle_encode_clip(clip, w, h, keep_recon=True, qp=24, gop=gop, cabac=1, me_range=8,
                                           slice_rows=rows, repeat_headers=1)
    with cx.Encoder(api.make_config(w, h, qp=24, gop=gop, cabac=1, me_range=8, max_clip_frames=n, slice_rows=rows,
                                    repeat_headers=1)) as enc:
        got, gsz = enc.encode_clip(clip)
        assert got == want and gsz.tolist() == sizes
        tail, _ = enc.encode_clip(clip[3:], first_frame_index=3)
    assert tail == want[sum(sizes[:3]):]
    dec = avdec.decode(tail)
    assert len(dec) == 6
    for p in range(3):
        assert np.array_equal(dec[-1][p], recs[-1][p])
    with cx.Encoder(api.make_config(w, h, qp=24, gop=gop, cabac=1, me_range=8, slice_rows=rows, repeat_headers=1)) as enc:
        frames = b"".join(enc.encode(*split_frame(clip[t], w, h, 0)) for t in range(n))
    assert frames == want


@pytest.mark.parametrize("cabac,rows", [(1, 0), (0, 0), (1, 3)])
def test_gpu_stream_through_the_golden_decoder(oracle, cabac, rows):
    """The CUDA encoder's stream, decoded by the golden model's decoder (no libavcodec), equals the CUDA encoder's own
    reconstruction."""
    w, h, n = 176, 144, 5
    clip = make_clip("synth", w, h, n)
    with cx.Encoder(api.make_config(w, h, qp=24, gop=3, cabac=cabac, slice_rows=rows)) as enc:
        stream, recs = b"", []
        for t in range(n):
            stream += enc.encode(*split_frame(clip[t], w, h, 0))
            recs.append(enc.debug_planes(2))
    dec = oracle.golden_decode(stream)
    assert len(dec) == n
    for r, d in zip(recs, dec):
        for p in range(3):
            assert np.array_equal(r[p], d[p])


# ---- intra4x4 extension (SURVEY 8f rank 2, I frames) -----------------------------------------------------------------
@pytest.mark.parametrize("cabac", [0, 1])
@pytest.mark.parametrize("kind,qp,rows", [("synth", 24, 0), ("noise", 12, 0), ("shift", 36, 0), ("synth", 30, 2), ("flat", 20, 0),
                                          ("noise", 1, 3)])
def test_intra4x4_every_stage_matches_oracle(oracle, kind, qp, rows, cabac):
    w, h, gop, n = 96, 80, 2, 4
    gold = oracle.Encoder(oracle.make_config(w, h, qp=qp, gop=gop, cabac=cabac, me_range=8, intra4x4=1, slice_rows=rows))
    with cx.Encoder(api.make_config(w, h, qp=qp, gop=gop, cabac=cabac, me_range=8, intra4x4=1, slice_rows=rows)) as enc:
        for t in range(n):
            y, c = content(kind, w, h, t)
            want, got = gold.encode(y, c), enc.encode(y, c)
            mbs = gold.mbs()
            mbi, nnz, coef = enc.debug_syntax()
            for k in ("type", "i16_mode", "chroma_mode", "cbp", "mv", "mvd"):
                assert np.array_equal(mbs[k], mbi[k]), "mb.%s frame %d" % (k, t)
            if gold.frame_is_i():
                i4 = mbs["type"] == 3
                assert np.array_equal(mbs["i4_mode"][i4], enc.debug_i4_modes()[i4]), "Intra4x4 modes frame %d" % t
            assert np.array_equal(mbs["nnz"], nnz[:, :27]), "nnz frame %d" % t
            assert np.array_equal(mbs["coef"], coef), "levels frame %d" % t
            for p, (a, b) in enumerate(zip(gold.recon(), enc.debug_planes(2))):
                assert np.array_equal(a, b), "recon plane %d frame %d" % (p, t)
            assert got == want, "bytestream frame %d" % t
    gold.close()


def test_intra4x4_clip_and_full_size(oracle):
    """clip mode == oracle at a small size; at 1080p the stream decodes (libavcodec) to the encoder's reconstruction and
    some macroblocks actually are Intra4x4."""
    w, h, n, gop = 96, 80, 7, 3
    clip = make_clip("synth", w, h, n)
    want, sizes, _ = oracle_encode_clip(clip, w, h, qp=24, gop=gop, cabac=1, me_range=8, intra4x4=1)
    with cx.Encoder(api.make_config(w, h, qp=24, gop=gop, cabac=1, me_range=8, max_clip_frames=n, intra4x4=1)) as enc:
        got, gsz = enc.encode_clip(clip)
    assert got == want and gsz.tolist() == sizes
    w, h = 1920, 1088
    clip = synth.synth_clip(w, h, [0, 1], 0).numpy()
    with cx.Encoder(api.make_config(w, h, qp=25, gop=60, cabac=1, intra4x4=1)) as enc:
        stream = enc.encode(*split_frame(clip[0], w, h, 0))
        ntype = (enc.debug_syntax()[0]["type"] == 3).sum()
        stream += enc.encode(*split_frame(clip[1], w, h, 0))
        last = enc.debug_planes(2)
    assert ntype > 0
    dec = avdec.decode(stream)
    for p in range(3):
        assert np.array_equal(dec[-1][p], last[p])


# ---- p_intra extension (SURVEY 8f rank 2, intra macroblocks inside P frames) -----------------------------------------
@pytest.mark.parametrize("cabac", [0, 1])
@pytest.mark.parametrize("kind,qp,rows", [("noise", 30, 0), ("noise", 12, 3), ("synth", 24, 0), ("shift", 36, 2), ("static", 30, 0)])
def test_p_intra_every_stage_matches_oracle(oracle, kind, qp, rows, cabac):
    w, h, gop, n = 96, 80, 4, 5
    gold = oracle.Encoder(oracle.make_config(w, h, qp=qp, gop=gop, cabac=cabac, me_range=8, p_intra=1, slice_rows=rows))
    intra_in_p = 0
    with cx.Encoder(api.make_config(w, h, qp=qp, gop=gop, cabac=cabac, me_range=8, p_intra=1, slice_rows=rows)) as enc:
        for t in range(n):
            y, c = content(kind, w, h, t)
            want, got = gold.encode(y, c), enc.encode(y, c)
            mbs = gold.mbs()
            mbi, nnz, coef = enc.debug_syntax()
            for k in ("type", "i16_mode", "chroma_mode", "cbp", "mv", "mvd"):
                assert np.array_equal(mbs[k], mbi[k]), "mb.%s frame %d" % (k, t)
            assert np.array_equal(mbs["nnz"], nnz[:, :27]), "nnz frame %d" % t
            assert np.array_equal(mbs["coef"], coef), "levels frame %d" % t
            for p, (a, b) in enumerate(zip(gold.recon(), enc.debug_planes(2))):
                assert np.array_equal(a, b), "recon plane %d frame %d" % (p, t)
            assert got == want, "bytestream frame %d" % t
            if not gold.frame_is_i():
                intra_in_p += int((mbs["type"] == 0).sum())
    gold.close()
    if kind == "noise":
        assert intra_in_p > 0, "the noise clip should exercise intra macroblocks in P frames"


def test_p_intra_clip_mode_and_decoders(oracle, monkeypatch):
    monkeypatch.setenv("CEDAR_B200_BINS_PER_MB", "4096")  # random-noise pictures need more than the clip-mode default
    w, h, n, gop = 96, 80, 9, 4
    clip = make_clip("noise", w, h, n)
    want, sizes, _ = oracle_encode_clip(clip, w, h, qp=28, gop=gop, cabac=1, me_range=8, p_intra=1)
    with cx.Encoder(api.make_config(w, h, qp=28, gop=gop, cabac=1, me_range=8, max_clip_frames=n, p_intra=1,
                                    gops_in_flight=2)) as enc:
        got, gsz = enc.encode_clip(clip)
    assert got == want and gsz.tolist() == sizes
    a, b = avdec.decode(got), oracle.golden_decode(got)
    assert len(a) == len(b) == n
    for x, y in zip(a, b):
        for p in range(3):
            assert np.array_equal(x[p], y[p])


# ---- queued per-frame mode and the multi-handle / multi-GPU pipeline (SURVEY 8b "queued mode", 8e) -----------------------
@pytest.mark.parametrize("cabac,n", [(1, 20), (0, 12), (1, 5), (1, 13)])
def test_queued_frame_mode_equals_oracle(oracle, cabac, n):
    """queue_gops = 2 with GOP 3: batches of 6 frames; encode_frame returns nothing for the first 12 calls, then frame
    t - 12; flush drains.  Frame by frame the bytes are the synchronous mode's, i.e. the golden model's."""
    w, h, gop = 96, 80, 3
    clip = make_clip("synth", w, h, n)
    want, sizes, _ = oracle_encode_clip(clip, w, h, qp=24, gop=gop, cabac=cabac, me_range=8)
    frames = []
    with cx.Encoder(api.make_config(w, h, qp=24, gop=gop, cabac=cabac, me_range=8, queue_gops=2)) as enc:
        for t in range(n):
            got = enc.encode(*split_frame(clip[t], w, h, 0))
            assert (len(got) == 0) == (t < 12), t
            if got:
                frames.append(got)
        while True:
            got = enc.flush()
            if not got:
                break
            frames.append(got)
        assert enc.flush() == b""
    assert [len(f) for f in frames] == sizes
    assert b"".join(frames) == want


@pytest.mark.parametrize("handles,batch,n", [(1, 1, 14), (2, 2, 20), (3, 1, 14), (2, 4, 7)])
def test_pipeline_equals_oracle(oracle, handles, batch, n):
    """Batches of whole GOPs round robin over several handles: the batches concatenate to the single stream (SPS/PPS only
    in front of frame 0, cedar.c:1058-1061), including a short last batch."""
    w, h, gop = 96, 80, 3
    clip = make_clip("synth", w, h, n)
    want, sizes, _ = oracle_encode_clip(clip, w, h, qp=24, gop=gop, cabac=1, me_range=8)
    with cx.Pipe(api.make_config(w, h, qp=24, gop=gop, cabac=1, me_range=8), None, handles, batch) as pipe:
        assert pipe.workers() == handles
        got, gsz = pipe.encode(clip)
    assert gsz == sizes and got == want


def test_pipeline_across_devices_equals_single_stream(oracle):
    """GOP-parallel across the GPUs of the box (every visible device; with one GPU the same device twice): batch b on
    worker b mod W, merged on the host == the golden model's single stream == one handle's stream (BASELINE.md gate 4)."""
    w, h, gop, n = 176, 144, 4, 40
    ndev = torch.cuda.device_count()
    devices = list(range(ndev)) if ndev > 1 else [0, 0]
    clip = make_clip("synth", w, h, n)
    want, sizes, _ = oracle_encode_clip(clip, w, h, qp=25, gop=gop, cabac=1, me_range=16)
    with cx.Pipe(api.make_config(w, h, qp=25, gop=gop, cabac=1), devices, 1, 1) as pipe:
        assert pipe.workers() == len(devices)
        got, gsz = pipe.encode(clip)
    assert gsz == sizes and got == want
    with cx.Encoder(api.make_config(w, h, qp=25, gop=gop, cabac=1, max_clip_frames=n)) as enc:
        one, _ = enc.encode_clip(clip)
    assert one == got


def test_pipeline_1080p_two_handles_equals_frame_mode():
    w, h, gop, n = 1920, 1088, 4, 16
    clip = synth.synth_clip(w, h, list(range(n)), 0).numpy()
    with cx.Pipe(api.make_config(w, h, qp=25, gop=gop, cabac=1), None, 2, 1) as pipe:
        got, gsz = pipe.encode(clip)
    with cx.Encoder(api.make_config(w, h, qp=25, gop=gop, cabac=1)) as enc:
        frames = [enc.encode(*split_frame(clip[t], w, h, 0)) for t in range(n)]
    assert [len(f) for f in frames] == gsz and b"".join(frames) == got


def test_stats_after_clip_encode_without_download(oracle):
    """cedar_b200_stats right after clip_encode (no clip_download in between) returns that encode's SSE."""
    w, h, n, gop = 96, 80, 5, 3
    clip = make_clip("synth", w, h, n)
    gold = oracle.Encoder(oracle.make_config(w, h, qp=24, gop=gop, me_range=8))
    want = []
    for t in range(n):
        gold.encode(*split_frame(clip[t], w, h, 0))
        want.append(gold.sse_y())
    gold.close()
    with cx.Encoder(api.make_config(w, h, qp=24, gop=gop, me_range=8, max_clip_frames=n)) as enc:
        enc.clip_input(n)[:] = clip
        enc.clip_upload(n)
        enc.clip_encode(n, 0)
        assert enc.sse_y(n).tolist() == want


def test_clip_mode_with_a_capacity_of_one_frame(oracle):
    """max_clip_frames = 1 is clip mode (it used to be mistaken for 'clip mode off')."""
    w, h = 64, 48
    clip = make_clip("synth", w, h, 1)
    want, sizes, _ = oracle_encode_clip(clip, w, h, qp=24, gop=1, me_range=8)
    with cx.Encoder(api.make_config(w, h, qp=24, gop=1, me_range=8, max_clip_frames=1)) as enc:
        got, gsz = enc.encode_clip(clip)
    assert got == want


@pytest.mark.parametrize("mbh", [1, 2, 17, 18, 34, 35, 52, 69])
@pytest.mark.parametrize("kind,qp", [("noise", 38), ("synth", 24)])
def test_deblocking_wavefront_across_cta_boundaries(oracle, mbh, kind, qp):
    """deblock_kernel cuts a picture into equally tall CTAs of at most 17 macroblock rows that hand rows over through
    global flags: every height around those cuts, strong (intra) and normal filtering, deblocked planes == golden model."""
    w, h = 80, 16 * mbh
    gold = oracle.Encoder(oracle.make_config(w, h, qp=qp, gop=2, cabac=0, me_range=4))
    with cx.Encoder(api.make_config(w, h, qp=qp, gop=2, cabac=0, me_range=4)) as enc:
        for t in range(3):
            y, c = content(kind, w, h, t)
            want, got = gold.encode(y, c), enc.encode(y, c)
            for p, (a, b) in enumerate(zip(gold.recon(), enc.debug_planes(2))):
                assert np.array_equal(a, b), "deblocked plane %d frame %d" % (p, t)
            assert got == want
    gold.close()


def test_queue_and_pipeline_edge_cases(oracle):
    """flush with nothing queued, close with frames still queued, a pipeline closed with unconsumed batches, an invalid
    configuration through the pipeline, a batch longer than the capacity: errors, never hangs."""
    import ctypes as C
    w, h, gop = 64, 48, 2
    cfg = api.make_config(w, h, qp=24, gop=gop, me_range=4, queue_gops=1)
    with cx.Encoder(cfg) as enc:
        assert enc.flush() == b""
    clip = make_clip("synth", w, h, 5)
    enc = cx.Encoder(cfg)
    for t in range(3):
        assert enc.encode(*split_frame(clip[t], w, h, 0)) == b""
    enc.close()  # frames still queued: dropped, no hang
    with pytest.raises(OSError):
        cx.Pipe(api.make_config(w, h, qp=99, gop=gop), None, 1, 1)
    with pytest.raises(OSError):
        cx.Pipe(api.make_config(w, h, qp=24, gop=gop, device=99), None, 1, 1)
    pipe = cx.Pipe(api.make_config(w, h, qp=24, gop=gop, me_range=4), None, 2, 1)
    buf = pipe.acquire()
    assert buf.shape[0] == gop
    with pytest.raises(OSError):
        pipe.submit(gop + 1)
    buf[:] = clip[:gop]
    pipe.submit(gop)
    buf = pipe.acquire()
    buf[:1] = clip[gop:gop + 1]
    pipe.submit(1)  # a short batch ends the stream: nothing may follow it
    with pytest.raises(RuntimeError):
        pipe.acquire()
    pipe.close()  # two batches never consumed
    want, _, _ = oracle_encode_clip(clip[:3], w, h, qp=24, gop=gop, cabac=1, me_range=4)
    with cx.Pipe(api.make_config(w, h, qp=24, gop=gop, me_range=4), None, 2, 1) as pipe:
        got, _ = pipe.encode(clip[:3])
    assert got == want
