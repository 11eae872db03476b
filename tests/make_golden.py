"""Regenerates the golden data under tests/golden/ from the REFERENCE decoder (oracle/_ref, built by oracle/Makefile from
the reference's sources), so that the tests compare with the reference wherever they run:
  streams.json            per generated stream: the reference's frame digests, FrameIds and cropped sizes; the digests
                          of the reference's own checked-in streams (copied to reference_streams/); the smoke clip
  api_reference.json      what the reference answered in tests/test_api_semantics.py
  full_size.json          the reference's `ref_decode -q` line of each full-size stream of tests/test_gpu_parity.py
  kat_fuzz_*.bin          per-trial digests of the reference's functions in the differential fuzz of oracle/ref_kat.c
Run where the reference's sources are: python tests/make_golden.py <reference source tree>"""
import json, os, shutil, subprocess, sys, tempfile
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from conftest import ROOT, STREAMS, DPB_STREAMS, make_stream, md5_frames
from checkers import decode_bytes

REF = sys.argv[1]
GOLDEN = os.path.join(ROOT, "tests", "golden")
tmp = tempfile.mkdtemp()


def frame_ids(frames):
    return [[f[0], f[1], f[2]] for f in frames]


out = {}
for name, w, h, args in STREAMS + DPB_STREAMS:
    data = open(make_stream(tmp, name, w, h, args), "rb").read()
    frames, _ = decode_bytes(data, "ref")
    out[name] = {"args": f"-W {w} -H {h} {args}", "bytes": len(data), "md5": md5_frames(frames), "frames": frame_ids(frames)}
refs = {}
os.makedirs(os.path.join(GOLDEN, "reference_streams"), exist_ok=True)
for f in ["finish-frame.264", "nal-ref-idc-0.264", "non-ref-dec-poc.264", "poc-out-of-order.264", "pos-frame-num-idr.264", "supp-nals.264", "zero-cropping.264"]:
    dst = os.path.join(GOLDEN, "reference_streams", f)
    shutil.copyfile(os.path.join(REF, "tests", f), dst)
    frames, _ = decode_bytes(open(dst, "rb").read(), "ref")
    refs[f] = md5_frames(frames)
out["_reference_streams"] = refs
import __graft_entry__
smoke = os.path.join(tmp, "smoke.264")
subprocess.run([os.path.join(ROOT, "tools", "gen264"), "-o", smoke] + __graft_entry__.SMOKE_ARGS, check=True, stderr=subprocess.DEVNULL)
out["_smoke"] = {"args": " ".join(__graft_entry__.SMOKE_ARGS), "md5": md5_frames(decode_bytes(open(smoke, "rb").read(), "ref")[0])}
json.dump(out, open(os.path.join(GOLDEN, "streams.json"), "w"), indent=1)
print("wrote", len(STREAMS + DPB_STREAMS), "streams")

import test_api_semantics as api
gold = {"borrowed": {}, "flush": {}, "unref": {}, "lost": {}}
for name, w, h, args in api.CASES:
    data = open(make_stream(tmp, name, w, h, args), "rb").read()
    for hold in (1, 3):
        frames, codes = api.decode_borrowing(data, "ref", hold)
        gold["borrowed"][f"{name}/{hold}"] = {"frames": api.digests(frames), "codes": codes}
data = open(make_stream(tmp, *api.STREAMS[6]), "rb").read()
for at in (7, 12):
    frames, codes = api.decode_borrowing(data, "ref", 0, flush_at=at)
    gold["flush"][str(at)] = {"frames": api.digests(frames), "codes": codes}
frames, allocs, _, _ = api.decode_with_allocator(data, "ref")
gold["allocator"] = {"frames": [[f[0], md5_frames([(0, 0, 0, f[1])])[0]] for f in frames], "allocs": sorted(set(allocs))}
for s in (api.STREAMS[2], api.STREAMS[6]):
    gold["unref"][s[0]] = api.decode_with_unref(open(make_stream(tmp, *s), "rb").read(), "ref")
for args, drop in api.LOST_CASES:
    path = os.path.join(tmp, "gap.264")
    subprocess.run([os.path.join(ROOT, "tools", "gen264"), "-o", path] + args.split(), check=True, stderr=subprocess.DEVNULL)
    nals = api._split_nals(open(path, "rb").read())
    ref, _ = decode_bytes(b"".join(n for k, n in enumerate(nals) if k not in drop), "ref")
    intact, _ = decode_bytes(b"".join(nals[:min(drop)]), "ref")
    n_before = max(0, len(intact) - 3)     # pictures complete and output-ordered before the first loss
    gold["lost"][args] = {"frames": frame_ids(ref), "md5_before": md5_frames(ref[:n_before])}
ref, codes = decode_bytes(api.sequence_changes_stream(tmp), "ref")
gold["sequence"] = {"frames": frame_ids(ref), "md5": md5_frames(ref), "codes": codes}
json.dump(gold, open(os.path.join(GOLDEN, "api_reference.json"), "w"), indent=1)
print("wrote api_reference.json")

import test_gpu_parity as parity
full = {}
for name, w, h, args in parity.FULL:
    r = subprocess.run([os.path.join(ROOT, "oracle", "_ref", "ref_decode"), make_stream(tmp, name, w, h, args), "-q"], capture_output=True, text=True, check=True)
    full[name] = r.stdout.strip().splitlines()[-1]
json.dump(full, open(os.path.join(GOLDEN, "full_size.json"), "w"), indent=1)
print("wrote full_size.json")

for what in ("fuzz", "residual", "deblock"):
    r = subprocess.run([os.path.join(ROOT, "oracle", "_ref", "ref_kat"), what, "--digests", os.path.join(GOLDEN, f"kat_fuzz_{what}.bin")], capture_output=True, text=True)
    assert r.returncode == 0 and ": ok" in r.stdout, r.stdout[-600:]
print("wrote kat_fuzz_*.bin")
shutil.rmtree(tmp)
