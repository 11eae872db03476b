"""Regenerates tests/golden/inter_fused.json: the REFERENCE decoder's frame digests (oracle/_ref, built by oracle/Makefile
from the reference's sources) of the inter streams of tests/test_inter_fused.py.
Run where the reference decoder is built: python tests/make_golden_inter_fused.py"""
import json, os, sys, tempfile
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from conftest import ROOT, make_stream, md5_frames
from checkers import decode_bytes
from test_inter_fused import FUSED_STREAMS

tmp = tempfile.mkdtemp()
fused = {}
for name, w, h, args in FUSED_STREAMS:
    data = open(make_stream(tmp, name, w, h, args), "rb").read()
    frames, _ = decode_bytes(data, "ref")
    fused[name] = {"args": f"-W {w} -H {h} {args}", "md5": md5_frames(frames)}
json.dump(fused, open(os.path.join(ROOT, "tests", "golden", "inter_fused.json"), "w"), indent=1)
print("wrote", len(fused), "streams")
