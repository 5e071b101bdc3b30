"""numpy model of the block-sum bound of me_kernel's search (kernels.cuh): on frames of the benchmark's synthetic clip
(1080p, a 1920 x 256 strip, R = 16, QP 25), the share of candidates whose bound key does not exceed the best key
(`vs final best`) or the key of the seeds (`vs seed`: the zero vector and the true background motion (+3, +2)).
Bounds over 16 groups of 16 pixels; quantised ones are what VABSDIFF4 evaluates four groups per instruction
(|A - B| >= 16 |A / 16 - B / 16| - 15).  The reference is the previous source frame, not the reconstruction.

    python tools/me_bound_model.py
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cedarx_h264_encoder_b200 import synth  # noqa: E402
W, H, R, qp, Y0, HS = 1920, 1088, 16, 25, 256, 256
lam = 1 << min(max((qp - 12) // 6, 0), 5)
bits = lambda d: 1 if d == 0 else 7 + 2 * (abs(d).bit_length() - 1)
nd = 2 * R + 1; mbw, mbh = W // 16, HS // 16
mvc = np.array([lam * bits(i - R) for i in range(nd)], np.int64)
rank = (np.arange(nd)[:, None] * nd + np.arange(nd)[None, :]).astype(np.int64); cmv = mvc[:, None] + mvc[None, :]
key = lambda c: ((np.maximum(c, 0).astype(np.int64) + cmv) << 15) | rank
for t in (1, 5, 31):
    cur = synth.synth_frame(W, H, t)[0].numpy().astype(np.int32)[Y0:Y0 + HS]
    refp = np.pad(synth.synth_frame(W, H, t - 1)[0].numpy().astype(np.int32), R, mode='edge')
    sad = np.zeros((mbh, mbw, nd, nd), np.int32); rowq = np.zeros_like(sad); subq = np.zeros_like(sad); rowx = np.zeros_like(sad)
    cr = cur.reshape(mbh, 16, mbw, 16).sum(axis=3)                       # [mby, row, mbx]
    cs = cur.reshape(mbh, 4, 4, mbw, 4, 4).sum(axis=(2, 5))              # 4x4 sub-block sums
    for oy in range(nd):
        for ox in range(nd):
            rf = refp[Y0 + oy:Y0 + oy + HS, ox:ox + W]
            sad[:, :, oy, ox] = np.abs(cur - rf).reshape(mbh, 16, mbw, 16).sum(axis=(1, 3))
            rr = rf.reshape(mbh, 16, mbw, 16).sum(axis=3)
            rowx[:, :, oy, ox] = np.abs(cr - rr).sum(axis=1)
            rowq[:, :, oy, ox] = 16 * np.abs(cr // 16 - rr // 16).sum(axis=1) - 240
            rs = rf.reshape(mbh, 4, 4, mbw, 4, 4).sum(axis=(2, 5))
            subq[:, :, oy, ox] = 16 * np.abs(cs // 16 - rs // 16).sum(axis=(1, 3)) - 240
    kb = key(sad); best = kb.reshape(mbh, mbw, -1).min(axis=2)[:, :, None, None]
    # seed-only threshold: min(zero vector, the vector that is the true background motion (+3,+2)) -- what the kernel's
    # co-located seed gives on background macroblocks from the second P frame of a GOP on
    seed = np.minimum(kb[:, :, R, R], kb[:, :, R + 2, R + 3])[:, :, None, None]
    for name, b in (("row sums exact", rowx), ("row sums /16 (VABSDIFF4)", rowq), ("4x4 sums /16 (VABSDIFF4)", subq),
                    ("max(row, 4x4) /16", np.maximum(rowq, subq))):
        print("t=%2d %-26s survive vs final best %.4f, vs seed %.4f" % (t, name, (key(b) <= best).mean(), (key(b) <= seed).mean()))
