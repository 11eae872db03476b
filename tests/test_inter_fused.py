"""The inter kernel's per-lane 4x4 reconstruction (transform, weighting and residual of a block in the lane that owns it:
luma on lanes 0-15, chroma on lanes 16-23) and its deblocking digests, against the CPU restatement and the reference's
digests (tests/golden/inter_fused.json, written by tests/make_golden_inter_fused.py), on inter streams that reach the
edges of those paths: both branches of the 8x8 dequantisation (qp / 6 below and above 4 at --qp 2 / --qp 50), only 4x4
or only 8x8 transforms, scaling matrices, the three weighting modes, dense chroma DC + AC, no skipped macroblocks, intra
macroblocks between inter ones.  The pictures
are 20x12 macroblocks: several 64-macroblock chunks of the inter kernel, whose first macroblock's left neighbour lies in
the chunk before."""
import json, os
import pytest
from conftest import ROOT, make_stream, md5_frames
from checkers import decode_bytes

FUSED_STREAMS = [
    ("fused_qp2",        20, 12, "-n 8 -s 51 --gop IPB --deblock 0 --t8x8 50 --qp 2 --refs 2 --density 90"),
    ("fused_qp50",       20, 12, "-n 8 -s 52 --gop IPB --deblock 0 --t8x8 50 --qp 50 --density 90"),
    ("fused_t8x8_0",     20, 12, "-n 8 -s 53 --gop IPB --deblock 0 --t8x8 0 --density 70"),
    ("fused_t8x8_100",   20, 12, "-n 8 -s 54 --gop IPB --deblock 0 --t8x8 100 --density 70"),
    ("fused_scaling",    20, 12, "-n 8 -s 55 --gop IPB --deblock 0 --t8x8 50 --scaling 3 --density 70"),
    ("fused_wp0",        20, 12, "-n 8 -s 56 --gop IPB --deblock 0 --wp 0 --refs 3 --density 60"),
    ("fused_wp1",        20, 12, "-n 8 -s 57 --gop IPB --deblock 0 --wp 1 --refs 3 --density 60"),
    ("fused_wp2",        20, 12, "-n 8 -s 58 --gop IPB --deblock 0 --wp 2 --temporal --density 60"),
    ("fused_dense_noskip", 20, 12, "-n 8 -s 59 --gop IPB --deblock 0 --density 90 --skip-pct 0 --wp 1"),
    ("fused_intra_mix",  20, 12, "-n 8 -s 60 --gop IPB --deblock 0 --intra-pct 30 --t8x8 50 --density 60"),
    ("fused_slices_dbk2", 20, 12, "-n 8 -s 61 --gop IPB --deblock 2 --slices 3 --intra-pct 15 --density 60"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,w,h,args", FUSED_STREAMS, ids=[s[0] for s in FUSED_STREAMS])
def test_inter_fused_matches_oracle_and_golden(workdir, name, w, h, args):
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "inter_fused.json")))[name]
    assert gold["args"] == f"-W {w} -H {h} {args}"
    data = open(make_stream(workdir, name, w, h, args), "rb").read()
    gpu, codes = decode_bytes(data, "gpu")
    assert md5_frames(gpu) == gold["md5"]
    port, pcodes = decode_bytes(data, "port")
    assert md5_frames(gpu) == md5_frames(port) and codes == pcodes
