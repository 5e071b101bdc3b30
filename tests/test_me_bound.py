"""The block-sum bound of the motion search (kernels.cuh, me_kernel's bound path): candidates whose quantised 4 x 4
sum bound exceeds the best key of the seeds are skipped, the others get their SAD, and a tile with more survivors than
its list holds searches exhaustively.  The motion vectors and the bytes must be the golden model's whatever the
content does to the bound; the work counters of the measurement build show which path each tile took."""
import numpy as np
import pytest
import torch

from common import content

try:
    import cedarx_h264_encoder_b200 as cx
    from cedarx_h264_encoder_b200 import api
except Exception:  # the CPU test below needs neither
    cx = api = None

gpu = pytest.mark.gpu
needs_cuda = pytest.mark.skipif(not torch.cuda.is_available(), reason="no CUDA device")


def quantised_bound(a, b):
    """16 * sum_g |floor(A_g / 16) - floor(B_g / 16)| - 240 over the sixteen 16-pixel groups of a 16 x 16 block pair"""
    A = a.reshape(4, 4, 4, 4).sum(axis=(1, 3)).astype(np.int64)
    B = b.reshape(4, 4, 4, 4).sum(axis=(1, 3)).astype(np.int64)
    return 16 * int(np.abs(A // 16 - B // 16).sum()) - 240


def test_quantised_bound_is_a_lower_bound_of_the_sad():
    r = np.random.default_rng(5)
    blocks = [r.integers(0, 256, (2, 16, 16)) for _ in range(2000)]
    # adversarial: every pixel of a group moves the same way (the exact group-sum bound is the SAD), and group sums
    # just below, at and above multiples of 16
    for _ in range(2000):
        a = np.repeat(np.repeat(r.integers(0, 240, (4, 4)), 4, 0), 4, 1)
        b = a + np.repeat(np.repeat(r.integers(0, 16, (4, 4)), 4, 0), 4, 1)
        blocks.append(np.stack([a, b]))
        k = r.integers(1, 255, (4, 4))
        a = np.repeat(np.repeat(k, 4, 0), 4, 1)
        b = a.copy()
        a[::4, ::4] += r.integers(-1, 2, (4, 4))
        b[::4, ::4] -= r.integers(-1, 2, (4, 4))
        blocks.append(np.stack([a, b]))
    for a, b in blocks:
        assert quantised_bound(a, b) <= int(np.abs(a.astype(np.int64) - b).sum())
    # the bound is reached: a group sum of 16 k against 16 k - 1 is |A - B| = 1 = 16 * 1 - 15
    a = np.full((16, 16), 16)
    b = a.copy()
    b[::4, ::4] -= 1
    assert quantised_bound(a, b) == int(np.abs(a - b).sum()) == 16


def _frames(kind, w, h, n):
    r = np.random.default_rng(11)
    ch = np.full((h // 2, w), 128, np.uint8)
    if kind == "permuted":  # pixels reversed inside each 4-pixel piece: 4 x 4 and row sums match, the SAD does not
        base = content("synth", w, h, 0)[0]
        return [(base, ch)] + [(base.reshape(h, w // 4, 4)[:, :, ::-1].reshape(h, w).copy(), ch) for _ in range(n - 1)]
    if kind == "tight":  # constant 4 x 4 groups that all move the same way between frames: the group-sum bound is the SAD
        g = r.integers(20, 200, (h // 4, w // 4))
        out = []
        for t in range(n):
            d = r.integers(0, 40, g.shape) if t else 0
            out.append((np.repeat(np.repeat(g + d, 4, 0), 4, 1).astype(np.uint8), ch))
        return out
    if kind == "edges":  # group sums at 16 k - 1, 16 k, 16 k + 1, content moving by (4, 4) pixels
        k = r.integers(1, 254, (h // 4 + 8, w // 4 + 8))
        out = []
        for t in range(n):
            big = np.repeat(np.repeat(k, 4, 0), 4, 1).astype(np.int32)
            big[::4, ::4] += r.integers(-1, 2, k.shape)
            y0 = 16 - 4 * t
            out.append((np.clip(big[y0:y0 + h, y0:y0 + w], 0, 255).astype(np.uint8), ch))
        return out
    if kind == "half_noise":  # left: fresh noise every frame (lists overflow), right: flat (the zero vector is the
        out = []              # only candidate whose key reaches the seed's)
        for t in range(n):
            y = np.full((h, w), 90, np.uint8)
            y[:, :w // 2] = r.integers(0, 256, (h, w // 2), dtype=np.uint8)
            out.append((y, ch))
        return out
    return [content(kind, w, h, t) for t in range(n)]


def _encode_against_golden(oracle, frames, w, h, me, qp=25, cabac=1):
    """encodes the frames with the measurement build; returns me_kernel's counters (MeShape::exec_count)"""
    gold = oracle.Encoder(oracle.make_config(w, h, qp=qp, gop=25, cabac=cabac, me_range=me))
    with cx.Encoder(api.make_config(w, h, qp=qp, gop=25, cabac=cabac, me_range=me)) as enc:
        enc.profile_enable(3)
        enc.profile_read(reset=True)
        for t, (y, c) in enumerate(frames):
            assert enc.encode(y, c) == gold.encode(y, c), "bytes of frame %d" % t
            assert np.array_equal(gold.mbs()["mv"], enc.debug_syntax()[0]["mv"]), "motion vectors of frame %d" % t
        cnt = np.zeros(520, np.uint64)
        assert enc.L.cedar_b200_debug_read(enc.h, 8, cnt.ctypes.data, cnt.nbytes) > 0
        enc.profile_enable(0)
    gold.close()
    return [int(v) for v in cnt[:5]]


@gpu
@needs_cuda
@pytest.mark.parametrize("kind", ["synth", "shift", "flat", "permuted", "tight", "edges"])
@pytest.mark.parametrize("me", [16, 8])
def test_bound_path_matches_golden(oracle, kind, me):
    w, h = 176, 144
    executed, bounded, sad, tiles, fallback = _encode_against_golden(oracle, _frames(kind, w, h, 4), w, h, me)
    assert tiles > 0 and bounded > 0 and executed > 0


@gpu
@needs_cuda
@pytest.mark.parametrize("me", [16, 32])
def test_list_overflow_searches_exhaustively(oracle, me):
    """noise on one half of a picture three tiles wide per half: those tiles overflow their lists, the others do not"""
    w, h = 384, 128
    executed, bounded, sad, tiles, fallback = _encode_against_golden(oracle, _frames("half_noise", w, h, 3), w, h, me)
    assert 0 < fallback < tiles, (fallback, tiles)
    assert sad > 0


@gpu
@needs_cuda
@pytest.mark.parametrize("me", [64, 1, 2, 3, 20, 32, 33, 47])
def test_every_geometry_with_clamped_windows(oracle, me):
    """the geometries of me_kernel (test_gpu_parity.test_me_ranges), on content whose best matches leave the picture:
    R 2..32 take the bound path, the others search exhaustively"""
    w, h = 208, 160
    frames = [content("shift", w, h, 3 * t) for t in range(3)]
    executed, bounded, sad, tiles, fallback = _encode_against_golden(oracle, frames, w, h, me)
    assert (tiles > 0) == (2 <= me <= 32)
    assert executed > 0
