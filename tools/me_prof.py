"""Diagnosis: cycles per tile of each phase of me_kernel (clock64 marks of a build with -DME_PROFILE) on a benchmark
workload.  Builds that library into a temporary directory (after the in-tree build, whose host objects it links), or
takes the one CEDAR_B200_LIB names.  Encodes the clip once to warm up, once measured; prints one JSON line.

    python tools/me_prof.py [--workload NAME] [--frames N] [--noise]

  cycles_per_tile  per phase, summed over the tiles of every P frame / tiles (a phase ends at a barrier, i.e. when
                   its slowest warp does):
    prologue   the tables, the current blocks, the seeds' vectors, and the window loads in flight
    staging    the window stores (copy 0 on the bound path, all four copies otherwise)
    seeds      the two seed candidates per macroblock, the quantised current sums and the block-sum table
    bound      the bound stage
    sad        the SAD stage of the listed candidates
    fallback   the exhaustive search (with the restaging of the shifted copies when a tile's list overflows)
    store      the motion vectors
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from cedarx_h264_encoder_b200 import api, synth  # noqa: E402

PHASES = ("prologue", "staging", "seeds", "bound", "sad", "fallback", "store")
SLOT = 480  # the counter slots past the CABAC context histogram: [480, 487) phases, [487] tiles


def build_profile_library(out_dir):
    pkg = os.path.join(ROOT, "cedarx_h264_encoder_b200")
    lib = os.path.join(out_dir, "libcedar_prof.so")
    subprocess.check_call(["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo",
                           "-std=c++17", "-Xcompiler", "-fPIC", "-DME_PROFILE", "-shared", "-o", lib,
                           os.path.join(pkg, "csrc", "encoder.cu"), os.path.join(pkg, "cedar_headers.o"),
                           os.path.join(pkg, "pipeline.o"), "--cudart", "static", "-lpthread"])
    return lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default=bench.DEFAULT_WORKLOAD)
    ap.add_argument("--frames", type=int, default=0, help="frames of the clip (0: the workload's)")
    ap.add_argument("--noise", action="store_true", help="uniform noise instead of the synthetic clip")
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        if not os.environ.get("CEDAR_B200_LIB"):
            os.environ["CEDAR_B200_LIB"] = build_profile_library(tmp)
        import cedarx_h264_encoder_b200 as cx
        w, h, fmt, n, gop, qp, me, cabac = bench.WORKLOADS[a.workload]
        n = a.frames or n
        enc = cx.Encoder(api.make_config(w, h, qp=qp, gop=gop, cabac=cabac, fmt=fmt, me_range=me, max_clip_frames=n))
        staging = torch.from_numpy(enc.clip_input(n))
        for i in range(0, n, 60):
            ids = list(range(i, min(n, i + 60)))
            if a.noise:
                g = torch.Generator().manual_seed(1234 + i)
                staging[i:i + len(ids)].copy_(torch.randint(0, 256, (len(ids), staging.shape[1]), generator=g,
                                                            dtype=torch.uint8))
            else:
                staging[i:i + len(ids)].copy_(synth.synth_clip(w, h, ids, fmt, device="cuda").cpu())
        enc.clip_upload(n)
        enc.clip_encode(n, 0)
        torch.cuda.synchronize()
        enc.profile_read(reset=True)  # clears the counters
        enc.clip_encode(n, 0)
        cnt = np.zeros(520, np.uint64)
        enc.L.cedar_b200_debug_read(enc.h, 8, cnt.ctypes.data, cnt.nbytes)
        tiles = int(cnt[SLOT + len(PHASES)])
        if not tiles:
            raise SystemExit("me_prof.py: no tile was counted; %s is not a -DME_PROFILE build"
                             % os.environ["CEDAR_B200_LIB"])
        per = {p: round(int(cnt[SLOT + i]) / tiles) for i, p in enumerate(PHASES)}
        out = {"workload": a.workload, "frames": n, "noise": a.noise, "gpu": torch.cuda.get_device_name(0),
               "tiles": tiles, "cycles_per_tile": per, "total": sum(per.values())}
        enc.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
