"""The reference itself, executed: kernel/cedar.c (unmodified, compiled by oracle/Makefile through oracle/refsim/kstub.h
from the reference's sources, which this repository does not contain) runs its CONFIG / ENCODE ioctls against a
software model of the video engine's registers; the macroblock engine behind the encode trigger (silicon in the
reference, cedar.c:1176) is the golden model.  Everything else in these streams -- start codes, SPS, PPS, slice headers,
the trailing-bits quirk, when parameter sets are sent, the GOP counter, the buffer sizes, the validation rules, the
register values -- is the reference's own code running.

CPU tests: golden model and product header writer against that.  GPU tests (-m gpu): the CUDA encoder through the C ABI
against that, frame by frame, and the product CLI against the reference's own userspace/h264enc.c (oracle/_ref/h264enc_sim).

The comparisons hold without the reference too: they compare against the answers it gave, recorded in tests/golden/
(headers.json, ref_streams.json, ref_answers.json), and where the reference is present (oracle/_ref/ prebuilt, or its
sources named by CEDAR_REFERENCE) they also check those recordings against it live.  Tests that inspect the driver's
own state or run the reference's own program need it and skip without it."""
import ctypes as C
import functools
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest
import torch

import refsim_lib as R
from common import content

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

LIVE = R.available()
live_only = pytest.mark.skipif(not LIVE, reason="runs the reference's own code: needs oracle/_ref/ or its sources (CEDAR_REFERENCE)")
needs_cuda = pytest.mark.skipif(not torch.cuda.is_available(), reason="no CUDA device")


@functools.lru_cache(maxsize=None)
def _golden(name):
    return json.load(open(os.path.join(HERE, "golden", name)))


def _run(kind, w, h, n, me=16, **kw):
    with R.Device(me_range=me) as d:
        assert d.config(R.make_config(w, h, **kw)) == 0
        return [d.encode(*content(kind, w, h, t)) for t in range(n)]


# ---------------------------------------------------------------------------------------------------------------------
# headers (SURVEY 8a H5-H8): reference code, live, against both restatements
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h", [(16, 16), (854, 480), (1280, 720), (1920, 1088), (1920, 1080), (3840, 2160), (4096, 2304)])
def test_sps_pps_equal_the_reference_writer(oracle, product_lib, w, h):
    from cedarx_h264_encoder_b200 import api
    gold = _golden("headers.json")
    for qp, cabac in ((24, 1), (25, 0), (1, 1), (47, 0)):
        sps = bytes.fromhex(gold["sps"]["%dx%d" % ((w + 15) & ~15, (h + 15) & ~15)])
        pps = bytes.fromhex(gold["pps"]["qp%02d_%s" % (qp, "cabac" if cabac else "cavlc")])
        if LIVE:
            nals = R.split_nals(_run("flat", w, h, 1, qp=qp, cabac=cabac)[0])
            assert (b"\x00\x00\x00\x01" + nals[0], b"\x00\x00\x00\x01" + nals[1]) == (sps, pps)
        assert oracle.write_sps(oracle.make_config(w, h, qp=qp, cabac=cabac)) == sps
        assert oracle.write_pps(oracle.make_config(w, h, qp=qp, cabac=cabac)) == pps
        assert api.write_sps(api.make_config(w, h, qp=qp, cabac=cabac)) == sps
        assert api.write_pps(api.make_config(w, h, qp=qp, cabac=cabac)) == pps


@live_only
def test_committed_header_vectors_are_what_the_reference_writes_today():
    """tests/golden/headers.json is generated (tests/golden/make_ref_headers.py); spot-check it against a live run."""
    gold = _golden("headers.json")
    nals = R.split_nals(_run("flat", 1920, 1088, 1, qp=25)[0])
    assert (b"\x00\x00\x00\x01" + nals[0]).hex(" ") == gold["sps"]["1920x1088"]
    assert (b"\x00\x00\x00\x01" + nals[1]).hex(" ") == gold["pps"]["qp25_cabac"]
    assert R.rbsp_bits(nals[2], 16) == gold["slice_bits"]["cabac"]["0"]


@live_only
@pytest.mark.parametrize("cabac", [0, 1])
def test_slice_headers_and_counters_over_two_gops(oracle, product_lib, cabac):
    """frame_p_count / frame_count as the driver keeps them (cedar.c:1193-1196), the picture type it derives
    (:1047-1050), parameter sets only before the first frame (:1058-1061), and the slice header bits per position."""
    from cedarx_h264_encoder_b200 import api
    gop, n = 5, 12
    with R.Device() as d:
        assert d.config(R.make_config(32, 32, gop=gop, cabac=cabac)) == 0
        for t in range(n):
            assert d.state("frame_p_count") == t % gop and d.state("frame_count") == t
            cur = d.state("reference_current")
            nals = R.split_nals(d.encode(*content("synth", 32, 32, t)))
            assert d.state("reference_current") == cur ^ 1  # cedar.c:1198-1201
            assert [x[0] for x in nals] == ([0x67, 0x68, 0x65] if t == 0 else [0x65 if t % gop == 0 else 0x41])
            p = t % gop
            nbits = 16 if p == 0 else (15 if cabac else 14)
            want = R.rbsp_bits(nals[-1], nbits)
            assert oracle.slice_header_bits(int(p == 0), p, cabac) == want
            assert api.slice_header_bits(int(p == 0), p, cabac) == want
            # PARA0: bit 8 = CABAC, bits 4-6 = slice type; PARA1: chroma QP offset 4, QP twice (cedar.c:1155-1168)
            para0, para1 = d.reg(R.ENC_BASE + R.PARA0), d.reg(R.ENC_BASE + R.PARA1)
            assert (para0 >> 8) & 1 == cabac and (para0 >> 4) & 7 == (0 if p == 0 else 1) and para0 >> 31 == 0
            assert para1 == (4 << 16) | (24 << 8) | 24
            assert d.reg(R.ENC_BASE + R.MEPARA) == 0x104


# ---------------------------------------------------------------------------------------------------------------------
# whole streams: reference driver + modelled engine == golden model on its own
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,w,h,n,qp,gop,cabac", [
    ("synth", 96, 80, 7, 24, 3, 1), ("synth", 96, 80, 7, 24, 3, 0), ("noise", 64, 48, 4, 1, 2, 1), ("noise", 64, 48, 4, 1, 2, 0),
    ("static", 96, 80, 6, 36, 31, 0), ("shift", 176, 144, 4, 47, 25, 1), ("synth", 854, 480, 3, 24, 25, 1), ("flat", 16, 16, 5, 12, 1, 1)])
def test_golden_model_stream_equals_reference_driver_stream(oracle, kind, w, h, n, qp, gop, cabac):
    want = next(c for c in _golden("ref_streams.json")["cases"]
                if (c["kind"], c["w"], c["h"], c["n"], c["qp"], c["gop"], c["cabac"]) == (kind, w, h, n, qp, gop, cabac))
    gold = oracle.Encoder(oracle.make_config(w, h, qp=qp, gop=gop, cabac=cabac, relax_gop=0))
    frames = [gold.encode(*content(kind, w, h, t)) for t in range(n)]
    gold.close()
    assert stream_record(frames) == {"sizes": want["sizes"], "sha256": want["sha256"]}
    if LIVE:
        ref = _run(kind, w, h, n, qp=qp, gop=gop, cabac=cabac)
        for t in range(n):
            assert frames[t] == ref[t], "frame %d" % t


def stream_record(frames):
    """What tests/golden/ keeps of a stream: the size of every frame and the SHA-256 of them all."""
    return {"sizes": [len(f) for f in frames], "sha256": hashlib.sha256(b"".join(frames)).hexdigest()}


def stream_fuzz_cases():
    """(w, h, config, content kind, frames, search range) of test_golden_model_stream_fuzz_equals_reference_driver_stream."""
    rng = np.random.default_rng(42)
    kinds = ["synth", "noise", "static", "shift", "flat"]
    cases = []
    for _ in range(24):
        w, h = int(rng.integers(8, 49)) * 2, int(rng.integers(8, 41)) * 2
        kw = dict(qp=int(rng.integers(1, 48)), gop=int(rng.integers(1, 32)), cabac=int(rng.integers(2)), fmt=0)
        kind, n, me = kinds[int(rng.integers(len(kinds)))], int(rng.integers(2, 6)), int(rng.choice([4, 8, 16]))
        cases.append((w, h, kw, kind, n, me))
    return cases


def test_golden_model_stream_fuzz_equals_reference_driver_stream(oracle):
    """The same comparison over seeded random small configurations: sizes that are not multiples of 16 (the driver pads
    to dst = ALIGN16, cedar.c:756-761), every QP, GOP lengths 1..31, both entropy coders, all content kinds.  NV12 only:
    the driver stores src_format and never programs it anywhere (cedar.c:793 is its last use), so a refsim run reads
    NV16 input as NV12 -- the NV16 path is the golden model's and the product's own (north star: "raw NV12/NV16")."""
    recorded = _golden("ref_answers.json")["stream_fuzz"]
    cases = stream_fuzz_cases()
    assert len(recorded) == len(cases)
    for (w, h, kw, kind, n, me), want in zip(cases, recorded):
        assert want["case"] == dict(w=w, h=h, kind=kind, n=n, me=me, **kw)
        gold = oracle.Encoder(oracle.make_config(w, h, relax_gop=0, me_range=me, **kw))
        frames = [gold.encode(*content(kind, w, h, t, kw["fmt"])) for t in range(n)]
        gold.close()
        assert stream_record(frames) == want["stream"], (w, h, kw, kind, me)
        if LIVE:
            with R.Device(me_range=me) as d:
                assert d.config(R.make_config(w, h, **kw)) == 0
                ref = [d.encode(*content(kind, w, h, t, kw["fmt"])) for t in range(n)]
            for t in range(n):
                assert frames[t] == ref[t], (w, h, kw, kind, me, t)


def test_committed_reference_stream_hashes(oracle):
    """The same comparison against committed hashes of the reference-driver streams (tests/golden/ref_streams.json), so it
    also holds where only the golden model can run."""
    gold = json.load(open(os.path.join(HERE, "golden", "ref_streams.json")))
    for c in gold["cases"]:
        enc = oracle.Encoder(oracle.make_config(c["w"], c["h"], qp=c["qp"], gop=c["gop"], cabac=c["cabac"]))
        frames = [enc.encode(*content(c["kind"], c["w"], c["h"], t)) for t in range(c["n"])]
        enc.close()
        assert [len(f) for f in frames] == c["sizes"], c
        assert hashlib.sha256(b"".join(frames)).hexdigest() == c["sha256"], c


# ---------------------------------------------------------------------------------------------------------------------
# configuration rules and buffer sizes (H2-H4)
# ---------------------------------------------------------------------------------------------------------------------
BAD = [dict(width=63), dict(height=47), dict(dst_width=70), dict(dst_height=50), dict(width=80, dst_width=64),
       dict(height=64, dst_height=48), dict(qp=0), dict(qp=48), dict(qp=-3), dict(fmt=2), dict(fmt=-1), dict(gop=0), dict(gop=32),
       dict(gop=-1)]
GOOD = [dict(), dict(qp=1), dict(qp=47), dict(gop=1), dict(gop=31), dict(fmt=1), dict(width=62, height=46), dict(cabac=0),
        dict(dst_width=128, dst_height=96)]


def _ref_config_rc(**kw):
    base = dict(width=64, height=48)
    base.update(kw)
    with R.Device() as d:
        return d.config(R.make_config(**base))


@pytest.mark.parametrize("kw", BAD + GOOD)
def test_config_validation_equals_the_reference_ioctl(oracle, product_lib, kw):
    """cedar_slashdev_ioctl_config (cedar.c:744-789), executed, against gm_open and cedar_b200_open (whose validation runs
    before any device is touched; relax_gop = 0 is the reference's rule)."""
    from cedarx_h264_encoder_b200 import api
    want = -22 if kw in BAD else 0
    if LIVE:
        assert _ref_config_rc(**kw) == want
    base = dict(width=64, height=48, relax_gop=0)
    base.update(kw)
    try:
        oracle.Encoder(oracle.make_config(**base)).close()
        got = 0
    except OSError as e:
        got = -e.errno
    assert got == want
    cfg, io, h = api.make_config(**base), api.CedarIO(), C.c_void_p()
    r = product_lib.cedar_b200_open(C.byref(cfg), C.byref(io), C.byref(h))
    if r == 0:
        product_lib.cedar_b200_close(h)
    assert r == want or (want == 0 and r == -19), "product %d, reference %d" % (r, want)  # -ENODEV: no GPU here


def _open_rc(make, base):
    try:
        make(base).close()
        return 0
    except OSError as e:
        return -e.errno


def config_fuzz_cases():
    """The configurations of test_config_validation_fuzz_equals_the_reference_ioctl."""
    rng = np.random.default_rng(20261018)
    def pick(good, bad):  # mostly a valid value, now and then one from beyond a limit
        v = bad if rng.random() < 0.12 else good
        return int(v[rng.integers(len(v))])
    cases = []
    for _ in range(300):
        w, h = pick((16, 62, 64, 100, 854, 1920, 4096), (1, 15, 17, 4097)), pick((16, 46, 48, 50, 480, 1088, 2304), (1, 15, 47, 4097))
        aw, ah = (w + 15) & ~15, (h + 15) & ~15
        cases.append(dict(width=w, height=h, qp=pick((1, 24, 47), (-1, 0, 48, 51, 100)), gop=pick((1, 2, 25, 31), (-1, 0, 32, 100)),
                          fmt=pick((0, 1), (-1, 2)), cabac=pick((0, 1), (0, 1)),
                          dst_width=pick((aw, aw, aw + 16, 4112), (w | 1, aw - 16, 0, aw + 8)),
                          dst_height=pick((ah, ah, ah + 16, 4112), (h | 1, ah - 16, 0, ah + 8))))
    return cases


def test_config_validation_fuzz_equals_the_reference_ioctl(oracle, product_lib):
    """The same three-way comparison over seeded random configurations around every limit of cedar.c:749-789 (most
    of them invalid: only the return value is compared, nothing is encoded).  Zero-sized pictures are left out: the
    reference's rules let them through and its allocator fails afterwards."""
    from cedarx_h264_encoder_b200 import api
    recorded = _golden("ref_answers.json")["config_fuzz"]
    cases = config_fuzz_cases()
    assert len(recorded) == len(cases)
    seen = {0: 0, -22: 0}
    for base, rec in zip(cases, recorded):
        assert rec["config"] == base
        want = rec["rc"]
        if LIVE:
            assert _ref_config_rc(**base) == want, base
        assert want in (0, -22), base
        seen[want] += 1
        assert _open_rc(lambda b: oracle.Encoder(oracle.make_config(relax_gop=0, **b)), base) == want, base
        cfg, io, hd = api.make_config(relax_gop=0, **base), api.CedarIO(), C.c_void_p()
        r = product_lib.cedar_b200_open(C.byref(cfg), C.byref(io), C.byref(hd))
        if r == 0:
            product_lib.cedar_b200_close(hd)
        assert r == want or (want == 0 and r in (-19, -12)), "%r: product %d, reference %d" % (base, r, want)
    assert seen[0] >= 60 and seen[-22] >= 60, seen  # the sweep reaches both sides


def header_fuzz_cases():
    """(w, h, gop, config) of test_header_fuzz_equals_the_reference_writer."""
    rng = np.random.default_rng(7)
    cases = []
    for _ in range(40):
        w, h = int(rng.integers(8, 41)) * 2, int(rng.integers(8, 31)) * 2
        kw = dict(qp=int(rng.integers(1, 48)), cabac=int(rng.integers(2)), profile=int(rng.choice([66, 77, 88, 100])),
                  level=int(rng.choice([10, 13, 30, 31, 40, 41, 42, 51])))
        gop = int(rng.integers(1, 32))
        cases.append((w, h, gop, kw))
    return cases


def test_header_fuzz_equals_the_reference_writer(oracle, product_lib):
    """SPS / PPS / first slice header for seeded random valid configurations (size, QP, profile_idc and level_idc as the
    caller passes them, entropy coder): reference driver (executed) == golden model == product writer."""
    from cedarx_h264_encoder_b200 import api
    recorded = _golden("ref_answers.json")["header_fuzz"]
    cases = header_fuzz_cases()
    assert len(recorded) == len(cases)
    for (w, h, gop, kw), rec in zip(cases, recorded):
        assert rec["case"] == dict(w=w, h=h, gop=gop, **kw)
        sps, pps, slice_bits = bytes.fromhex(rec["sps"]), bytes.fromhex(rec["pps"]), rec["slice_bits"]
        if LIVE:
            with R.Device() as d:
                assert d.config(R.make_config(w, h, gop=gop, **kw)) == 0
                nals = R.split_nals(d.encode(*content("flat", w, h, 0)))
            assert (b"\x00\x00\x00\x01" + nals[0], b"\x00\x00\x00\x01" + nals[1], R.rbsp_bits(nals[2], 16)) == (sps, pps, slice_bits)
        for mod in (oracle, api):
            c = mod.make_config(w, h, gop=gop, **kw)
            assert mod.write_sps(c) == sps and mod.write_pps(c) == pps, (w, h, kw)
            assert mod.slice_header_bits(1, 0, kw["cabac"]) == slice_bits


@live_only
def test_second_config_is_rejected_and_encode_needs_config():
    with R.Device() as d:
        assert d.L.refsim_ioctl(R.IOCTL_ENCODE, None) == -22  # cedar.c:1039-1043
        assert d.config(R.make_config(64, 48)) == 0
        assert d.config(R.make_config(64, 48)) == -22         # cedar.c:744-747
        assert d.L.refsim_ioctl(0x777, None) == -1            # cedar.c:1222-1225


@live_only
@pytest.mark.parametrize("w,h", [(854, 480), (1280, 720), (1920, 1088), (3840, 2160)])
def test_buffer_sizes_of_the_reference(w, h):
    """cedar_buffers_init / cedar_reference_frame_init (cedar.c:500-538, 605-704), executed; SURVEY 8a row H4."""
    def al(x, a):
        return (x + a - 1) // a * a
    W, H = al(w, 16), al(h, 16)
    with R.Device() as d:
        cfg = R.make_config(w, h)
        assert d.config(cfg) == 0
        assert cfg.input_luma_size == al(w * h, 4096) == d.state("input_luma_size")
        assert cfg.input_chroma_size == al(w * h // 2, 4096)
        assert cfg.bytestream_size == 1 << 20
        assert d.state("ref_luma_size") == al(W, 32) * al(H, 64)
        assert d.state("ref_chroma_size") == al(W, 32) * al(H, 128) // 2
        assert d.state("ref_subpic_size") == d.state("ref_luma_size") // 2
        assert d.state("mb_info_size") == W * 8
        assert d.state("mv_buffer_size") == al(W // 16, 4) * (H // 16) * 8
        assert (cfg.thumbnail, cfg.thumb_luma_size) == (0, 0)
        assert d.state("src_stride_mb") == d.state("src_width_mb") == W // 16
    assert d.L.refsim_dma_live() == 0, "release frees every buffer (cedar.c:706-730)"


# ---------------------------------------------------------------------------------------------------------------------
# the reference's own CLI, end to end
# ---------------------------------------------------------------------------------------------------------------------
def _write_clip(path, w, h, n):
    with open(path, "wb") as f:
        for t in range(n):
            y, c = content("synth", w, h, t)
            f.write(y.tobytes())
            f.write(c.tobytes())


@live_only
def test_reference_cli_end_to_end_equals_golden_cli(oracle, tmp_path):
    """BASELINE.json configs[0]: 854x480 NV12, 30 frames, the reference's defaults (QP 24, GOP 25, CABAC) through the
    reference's unmodified userspace/h264enc.c + kernel/cedar.c == the golden model's CLI, byte for byte."""
    w, h, n = 854, 480, 30
    src, a, b = str(tmp_path / "in.nv12"), str(tmp_path / "ref.264"), str(tmp_path / "gold.264")
    _write_clip(src, w, h, n)
    r = subprocess.run([R.CLI, src, str(w), str(h), a], capture_output=True, timeout=300)  # bytes: keep the \r
    assert r.returncode == 0, r.stderr
    assert r.stdout.count(b"\rFrame") == n and b"Input Y: %dbytes at 0x" % ((w * h + 4095) // 4096 * 4096) in r.stdout
    subprocess.run([os.path.join(ROOT, "oracle", "golden_enc"), src, str(w), str(h), b], check=True, capture_output=True, timeout=300)
    assert open(a, "rb").read() == open(b, "rb").read()
    assert os.stat(a).st_mode & 0o777 == 0o644 & ~_umask()
    # usage: exactly four arguments, else the usage line and -1 (userspace/h264enc.c:141-144)
    r = subprocess.run([R.CLI, src, str(w)], capture_output=True, text=True)
    assert r.returncode == 255 and r.stdout.startswith("Usage: ")


def test_reference_cli_bound_to_the_product_has_no_cpu_path(tmp_path):
    """oracle/_ref/h264enc_b200 = userspace/h264enc.c, unmodified, with its /dev/cedar_dev calls bound to libcedar_b200.so
    (oracle/refsim/b200_shim.c).  Without a GPU the CONFIG ioctl fails with ENODEV and the program ends the way the
    reference does when its ioctl fails (userspace/h264enc.c:68-73,151-153); the usage line is the reference's."""
    import torch
    if not os.path.exists(R.CLI_B200):
        pytest.skip("oracle/_ref/h264enc_b200 is built where the reference sources are")
    r = subprocess.run([R.CLI_B200, "a", "b"], capture_output=True, text=True)
    assert r.returncode == 255 and r.stdout.startswith("Usage: ")
    if torch.cuda.is_available():
        pytest.skip("GPU present: see test_unmodified_reference_cli_on_the_product_library")
    src = tmp_path / "in.nv12"
    src.write_bytes(bytes(96 * 80 * 3 // 2))
    r = subprocess.run([R.CLI_B200, str(src), "96", "80", str(tmp_path / "o.264")], capture_output=True, text=True)
    assert r.returncode == 255
    assert "CEDAR_IOCTL_CONFIG failed: No such device" in r.stderr and "no CPU fallback" in r.stderr


def _umask():
    m = os.umask(0)
    os.umask(m)
    return m


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the product through its C ABI against the reference driver, call for call
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@needs_cuda
@pytest.mark.parametrize("kind,w,h,n,qp,gop,cabac", [("synth", 854, 480, 27, 24, 25, 1), ("synth", 96, 80, 8, 24, 3, 0),
                                                   ("noise", 64, 48, 4, 1, 2, 1), ("shift", 176, 144, 5, 30, 31, 1),
                                                   ("synth", 1920, 1088, 3, 25, 25, 1)])
def test_product_equals_reference_driver_frame_by_frame(kind, w, h, n, qp, gop, cabac):
    """ioctl(CEDAR_IOCTL_CONFIG) / ioctl(CEDAR_IOCTL_ENCODE) on the reference driver vs cedar_b200_open /
    cedar_b200_encode_frame: same return value (bytes in the bytestream buffer) and same bytes, every frame, with the
    same config struct fields and the same buffer sizes reported back."""
    import cedarx_h264_encoder_b200 as cx
    from cedarx_h264_encoder_b200 import api
    rec = _golden("ref_answers.json")["frame_by_frame"]["%s_%dx%d_%df_qp%d_gop%d_%s" % (kind, w, h, n, qp, gop,
                                                                                       "cabac" if cabac else "cavlc")]
    d = R.Device() if LIVE else None
    try:
        if d:
            rcfg = R.make_config(w, h, qp=qp, gop=gop, cabac=cabac)
            assert d.config(rcfg) == 0
            assert (rcfg.input_luma_size, rcfg.input_chroma_size) == (rec["input_luma_size"], rec["input_chroma_size"])
        with cx.Encoder(api.make_config(w, h, qp=qp, gop=gop, cabac=cabac, relax_gop=0)) as enc:
            assert enc.io.input_luma_size == rec["input_luma_size"] and enc.io.input_chroma_size == rec["input_chroma_size"]
            for t in range(n):
                y, c = content(kind, w, h, t)
                got = enc.encode(y, c)
                assert len(got) == rec["sizes"][t] and hashlib.sha256(got).hexdigest() == rec["sha256"][t], "frame %d" % t
                if d:
                    assert got == d.encode(y, c), "frame %d" % t
    finally:
        if d:
            d.close()


@pytest.mark.gpu
@needs_cuda
def test_product_cli_equals_reference_cli(tmp_path):
    """h264enc <in> <w> <h> <out>: the product CLI and the reference's own program (in simulation) write the same file
    and print the same progress lines ("\\rFrame %5d: %5dbytes", userspace/h264enc.c:194)."""
    w, h, n = 854, 480, 30
    rec = _golden("ref_answers.json")["cli_854x480_30f"]
    src, a, b = str(tmp_path / "in.nv12"), str(tmp_path / "ref.264"), str(tmp_path / "b200.264")
    _write_clip(src, w, h, n)
    exe = os.path.join(ROOT, "cedarx_h264_encoder_b200", "h264enc")
    r2 = subprocess.run([exe, src, str(w), str(h), b], capture_output=True, timeout=300)
    assert r2.returncode == 0, r2.stderr
    got = open(b, "rb").read()
    assert len(got) == sum(rec["sizes"]) and hashlib.sha256(got).hexdigest() == rec["sha256"]
    prog = lambda s: [x for x in s.split(b"\r") if x.startswith(b"Frame")]  # noqa: E731
    assert [x.rstrip(b"\n") for x in prog(r2.stdout)] == [b"Frame %5d: %5dbytes" % (i, s) for i, s in enumerate(rec["sizes"])]
    if LIVE:
        r1 = subprocess.run([R.CLI, src, str(w), str(h), a], capture_output=True, timeout=300)
        assert r1.returncode == 0
        assert open(a, "rb").read() == got
        assert prog(r1.stdout) == prog(r2.stdout)


@live_only
@pytest.mark.gpu
def test_unmodified_reference_cli_on_the_product_library(tmp_path):
    """The drop-in boundary, executed: the reference's own userspace/h264enc.c -- not a line changed, compiled from
    /root/reference by oracle/Makefile -- with open / ioctl / mmap on /dev/cedar_dev bound to the product's C ABI
    (oracle/refsim/b200_shim.c, the binding of INTEGRATION.md section 2) writes the same file and prints the same
    progress lines as the same program on the reference's own driver in simulation."""
    if not os.path.exists(R.CLI_B200):
        pytest.fail("oracle/_ref/h264enc_b200 missing: it is built next to h264enc_sim and travels with it")
    w, h, n = 176, 144, 28
    src, a, b = str(tmp_path / "in.nv12"), str(tmp_path / "ref.264"), str(tmp_path / "b200.264")
    _write_clip(src, w, h, n)
    r1 = subprocess.run([R.CLI, src, str(w), str(h), a], capture_output=True, timeout=300)
    r2 = subprocess.run([R.CLI_B200, src, str(w), str(h), b], capture_output=True, timeout=300)
    assert r1.returncode == 0 and r2.returncode == 0, r2.stderr
    assert open(a, "rb").read() == open(b, "rb").read()
    prog = lambda s: [x for x in s.split(b"\r") if x.startswith(b"Frame")]  # noqa: E731
    assert prog(r1.stdout) == prog(r2.stdout) and len(prog(r2.stdout)) == n
    assert b"Time spent" in r2.stderr  # cedar_b200_close at exit, like the driver's release (kernel/cedar.c:706-730)
