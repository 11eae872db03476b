"""Pins the oracle: the host parser + record ABI + CPU restatement (oracle/liboracle_dec.so) must give
the reference decoder's exact YUV on generated streams, and both must match the committed golden
digests, FrameIds and cropped sizes (tests/golden/streams.json, produced by tests/make_golden.py from the reference)."""
import json, os
import pytest
from conftest import ROOT, STREAMS, DPB_STREAMS, make_stream, md5_frames
from checkers import decode_bytes

GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "streams.json")))


@pytest.mark.parametrize("name,w,h,args", STREAMS + DPB_STREAMS, ids=[s[0] for s in STREAMS + DPB_STREAMS])
def test_port_matches_reference_and_golden(workdir, name, w, h, args):
    data = open(make_stream(workdir, name, w, h, args), "rb").read()
    port, _ = decode_bytes(data, "port")
    assert md5_frames(port) == GOLD[name]["md5"], "oracle port differs from the golden reference output"
    assert [[f[0], f[1], f[2]] for f in port] == GOLD[name]["frames"]   # FrameId, cropped size


def test_reference_header_streams(workdir):
    """The reference's own checked-in streams (DPB / POC / cropping corner cases, 1x1 macroblock), copied to
    tests/golden/reference_streams/, against the digests of the reference's output."""
    d = os.path.join(ROOT, "tests", "golden", "reference_streams")
    for name, want in GOLD["_reference_streams"].items():
        frames, _ = decode_bytes(open(os.path.join(d, name), "rb").read(), "port")
        assert md5_frames(frames) == want, name
