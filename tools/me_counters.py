"""Work counters of me_kernel on a benchmark workload: the measurement build (profile mode 3) encodes the clip once and
reports what the motion search did.  Prints one JSON line.

    python tools/me_counters.py [--workload NAME] [--frames N] [--noise]

  executed_over_algorithmic  VABSDIFF4 lane-instructions executed (block sums, bounds, SADs) / 64 per candidate
  bounded_frac               candidates whose block-sum bound was evaluated / all candidates
  sad_frac                   candidates that reached the SAD stage / all candidates
  fallback_tiles             bound-path tiles whose candidate list overflowed and that searched exhaustively
  me_kernel_ms               standalone time of me_kernel over the clip (profile mode 2, every kernel on one stream)
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import cedarx_h264_encoder_b200 as cx  # noqa: E402
from cedarx_h264_encoder_b200 import api, synth  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default=bench.DEFAULT_WORKLOAD)
    ap.add_argument("--frames", type=int, default=0, help="frames of the clip (0: the workload's)")
    ap.add_argument("--noise", action="store_true", help="uniform noise instead of the synthetic clip")
    a = ap.parse_args()
    w, h, fmt, n, gop, qp, me, cabac = bench.WORKLOADS[a.workload]
    n = a.frames or n
    enc = cx.Encoder(api.make_config(w, h, qp=qp, gop=gop, cabac=cabac, fmt=fmt, me_range=me, max_clip_frames=n))
    staging = torch.from_numpy(enc.clip_input(n))
    for i in range(0, n, 60):
        ids = list(range(i, min(n, i + 60)))
        if a.noise:
            g = torch.Generator().manual_seed(1234 + i)
            staging[i:i + len(ids)].copy_(torch.randint(0, 256, (len(ids), staging.shape[1]), generator=g, dtype=torch.uint8))
        else:
            staging[i:i + len(ids)].copy_(synth.synth_clip(w, h, ids, fmt, device="cuda").cpu())
    enc.clip_upload(n)
    enc.clip_encode(n, 0)
    enc.clip_download(n)
    enc.profile_enable(2)
    enc.profile_read(reset=True)
    enc.clip_encode(n, 0)
    prof = enc.profile_read(reset=True)
    enc.profile_enable(3)
    enc.profile_read(reset=True)
    enc.clip_encode(n, 0)
    cnt = np.zeros(520, np.uint64)
    enc.L.cedar_b200_debug_read(enc.h, 8, cnt.ctypes.data, cnt.nbytes)
    enc.profile_read(reset=True)
    enc.profile_enable(0)
    torch.cuda.synchronize()
    W16, H16 = (w + 15) // 16, (h + 15) // 16
    p_frames = n - -(-n // gop)
    cands = p_frames * W16 * H16 * (2 * me + 1) ** 2
    out = {"workload": a.workload, "frames": n, "noise": a.noise, "gpu": torch.cuda.get_device_name(0),
           "me_kernel_ms": round(prof.get("me_kernel", (0.0, 0))[0], 3),
           "executed_over_algorithmic": int(cnt[0]) / (64.0 * cands),
           "bounded_frac": int(cnt[1]) / cands, "sad_frac": int(cnt[2]) / cands,
           "bound_tiles": int(cnt[3]), "fallback_tiles": int(cnt[4])}
    enc.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
