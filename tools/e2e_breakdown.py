"""Where the end-to-end figure loses against the device-resident one: three handles on three host threads over the
benchmark clip (1920x1080 NV12, 600 frames, GOP 60, QP 25), the step body varied.

    python tools/e2e_breakdown.py [steps] [out.jsonl] [handles] [bodies, comma separated]

`steps` clips in all, dealt round robin to the handles like bench.py does (20 steps over three handles: 7 + 7 + 6).

  encode            clip_encode back to back, nothing else (bench.py's `value`)
  encode+sync       clip_encode, then the host waits for it (cedar_b200_stats synchronises the handle's stream)
  upload+encode     clip_upload + clip_encode, no wait in between the clips
  encode+download   clip_encode + clip_download (waits, 10.6 MB device -> host)
  e2e               clip_upload + clip_encode + clip_download (bench.py's `e2e`)

Wall clock around issue + synchronize, warm; frames/s.
"""
import json
import os
import sys
import threading
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import cedarx_h264_encoder_b200 as cx  # noqa: E402
from cedarx_h264_encoder_b200 import api, synth  # noqa: E402

w, h, gop, qp, me, n = 1920, 1080, 60, 25, 16, 600


def make():
    enc = cx.Encoder(api.make_config(w, h, qp=qp, gop=gop, cabac=1, me_range=me, max_clip_frames=n))
    staging = torch.from_numpy(enc.clip_input(n))
    for i in range(0, n, 20):
        part = synth.synth_clip(w, h, list(range(i, min(n, i + 20))), 0, device="cuda")
        staging[i:i + len(part)].copy_(part)
    torch.cuda.synchronize()
    enc.clip_upload(n)
    enc.clip_encode(n, 0)
    enc.clip_download(n)
    return enc


def run(encs, body, steps):
    def work(i):
        for _ in range(i, steps, len(encs)):
            body(encs[i])
    for e in encs:
        body(e)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    th = [threading.Thread(target=work, args=(i,)) for i in range(len(encs))]
    [t.start() for t in th]
    [t.join() for t in th]
    torch.cuda.synchronize()
    return n * steps / (time.perf_counter() - t0)


def main():
    steps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    nh = int(sys.argv[3]) if len(sys.argv) > 3 else 3
    only = sys.argv[4].split(",") if len(sys.argv) > 4 else None
    encs = [make() for _ in range(nh)]
    bodies = {
        "encode": lambda e: e.clip_encode(n, 0),
        "encode+sync": lambda e: (e.clip_encode(n, 0), e.sse_y(1)),
        "upload+encode": lambda e: (e.clip_upload(n), e.clip_encode(n, 0)),
        "encode+download": lambda e: (e.clip_encode(n, 0), e.clip_download(n)),
        "e2e": lambda e: (e.clip_upload(n), e.clip_encode(n, 0), e.clip_download(n)),
    }
    res = {"steps": steps, "handles": nh}
    for name, body in bodies.items():
        if only and name not in only:
            continue
        res[name] = round(run(encs, body, steps))
        print("%-16s %6d frames/s" % (name, res[name]), file=sys.stderr, flush=True)
    for e in encs:
        e.close()
    print(json.dumps(res))
    if len(sys.argv) > 2:
        with open(sys.argv[2], "a") as f:
            f.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
