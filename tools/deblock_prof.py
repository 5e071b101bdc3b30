"""Diagnosis: per-phase clock64 timing of the luma deblocking warp (needs tools/libcedar_prof.so built with
-DDB_PROFILE)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cedarx_h264_encoder_b200 import api, synth
api.LIB_NAME = "../tools/libcedar_prof.so"
import cedarx_h264_encoder_b200 as cx
w, h, n, gop = 1920, 1088, 4, 60
enc = cx.Encoder(api.make_config(w, h, qp=25, gop=gop, cabac=0, max_clip_frames=n))
clip = synth.synth_clip(w, h, list(range(n))).numpy()
enc.encode_clip(clip)
enc.close()
