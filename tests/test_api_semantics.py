"""API behaviour beyond the plain decode loop, compared between the reference and our host code (CPU backend):
borrowed frames (edge264_get_frame(borrow=1) / edge264_return_frame, reference edge264.c:365-414), flush in the middle
of a stream (edge264.c:261-270), and the sequence of return codes of edge264_decode_NAL.  What the reference answered
is recorded in tests/golden/api_reference.json (tests/make_golden.py)."""
import ctypes, errno, hashlib, json, os
import pytest
from conftest import ROOT, STREAMS, make_stream
from checkers import load, Edge264Frame, _frame_bytes



@pytest.fixture(scope="module")
def gold():
    return json.load(open(os.path.join(ROOT, "tests", "golden", "api_reference.json")))


def digests(frames):
    return [[f[0], hashlib.md5(f[3]).hexdigest()] for f in frames]


def decode_borrowing(data, backend, hold, flush_at=None):
    lib = load(backend)
    buf = ctypes.create_string_buffer(data, len(data) + 64)
    base = ctypes.addressof(buf); end = base + len(data)
    dec = lib.edge264_alloc(0, None, None, 0, None, None, None)
    assert dec
    nal = base + 3 + (1 if data[2] == 0 else 0)
    held, out, codes, f, n_nal, drained = [], [], [], Edge264Frame(), 0, False
    while True:
        sc = lib.edge264_find_start_code(nal, end, 0) if nal < end else end
        before = len(out) + len(held)
        res = lib.edge264_decode_NAL(dec, nal, sc, None, None)
        if nal >= end:
            drained = True
        while lib.edge264_get_frame(dec, ctypes.byref(f), 1) == 0:
            # remember where the samples live and what they look like now; they must be unchanged when we give them back
            held.append((f.FrameId, f.width_Y, f.height_Y, _frame_bytes(f), f.return_arg, Edge264Frame.from_buffer_copy(bytes(f))))
            while len(held) > hold:
                fid, w, h, snap, arg, fr = held.pop(0)
                assert _frame_bytes(fr) == snap, "a borrowed frame changed while it was held"
                out.append((fid, w, h, snap))
                lib.edge264_return_frame(dec, arg)
        if res == errno.ENOBUFS:
            if len(out) + len(held) == before:
                if not held:
                    break
                fid, w, h, snap, arg, fr = held.pop(0)      # the decoder is out of frame buffers: hand one back
                assert _frame_bytes(fr) == snap
                out.append((fid, w, h, snap)); lib.edge264_return_frame(dec, arg)
            continue
        codes.append(res)
        n_nal += 1
        if flush_at is not None and n_nal == flush_at:
            for fid, w, h, snap, arg, fr in held:
                out.append((fid, w, h, snap)); lib.edge264_return_frame(dec, arg)
            held = []
            lib.edge264_flush(dec)
        if res in (errno.ENOTSUP, errno.EBADMSG):
            res = 0
        nal = sc + 3 if sc + 3 < end else end
        if res != 0 or drained:
            break
    for fid, w, h, snap, arg, fr in held:
        assert _frame_bytes(fr) == snap
        out.append((fid, w, h, snap)); lib.edge264_return_frame(dec, arg)
    d = ctypes.c_void_p(dec)
    lib.edge264_free(ctypes.byref(d))
    return out, codes


CASES = [STREAMS[6], STREAMS[8], STREAMS[9]]   # I P B B streams: frames leave out of decoding order


@pytest.mark.parametrize("name,w,h,args", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("hold", [1, 3])
def test_borrowed_frames_match_reference(workdir, gold, name, w, h, args, hold):
    data = open(make_stream(workdir, name, w, h, args), "rb").read()
    plain, _ = decode_borrowing(data, "port", 0)
    ours, codes = decode_borrowing(data, "port", hold)
    assert [(f[0], f[3]) for f in ours] == [(f[0], f[3]) for f in plain], "holding frames changed the output"
    ref = gold["borrowed"][f"{name}/{hold}"]
    assert ref["frames"] == digests(ours)
    assert ref["codes"] == codes, "edge264_decode_NAL return codes differ from the reference's"


def test_flush_mid_stream_matches_reference(workdir, gold):
    name, w, h, args = STREAMS[6]
    data = open(make_stream(workdir, name, w, h, args), "rb").read()
    for at in (7, 12):
        ours, codes = decode_borrowing(data, "port", 0, flush_at=at)
        ref = gold["flush"][str(at)]
        assert ref["codes"] == codes
        assert ref["frames"] == digests(ours)


UNREF = ctypes.CFUNCTYPE(None, ctypes.c_int, ctypes.c_void_p)


def decode_with_unref(data, backend):
    """Every edge264_decode_NAL gets an unref callback; returns [(return code, callback calls as (ret, arg))] per NAL."""
    lib = load(backend)
    buf = ctypes.create_string_buffer(data, len(data) + 64)
    base = ctypes.addressof(buf); end = base + len(data)
    dec = lib.edge264_alloc(0, None, None, 0, None, None, None)
    nal = base + 3 + (1 if data[2] == 0 else 0)
    calls, log, f, k = [], [], Edge264Frame(), 0
    cb = UNREF(lambda ret, arg: calls.append((ret, arg)))
    while nal < end:
        sc = lib.edge264_find_start_code(nal, end, 0)
        k += 1
        n0 = len(calls)
        res = lib.edge264_decode_NAL(dec, nal, sc, cb, ctypes.c_void_p(k))
        while lib.edge264_get_frame(dec, ctypes.byref(f), 0) == 0:
            pass
        if res == errno.ENOBUFS:
            k -= 1
            continue
        log.append((res, calls[n0:]))
        nal = sc + 3 if sc + 3 < end else end
    d = ctypes.c_void_p(dec)
    lib.edge264_free(ctypes.byref(d))
    return log


def test_unref_callback_matches_reference(workdir, gold):
    """n_threads = 0: the reference calls unref_cb(ret, arg) exactly once before edge264_decode_NAL returns, for slices and
    for every other NAL (edge264.c:356-357, edge264_headers.c:497-498)."""
    for name, w, h, args in (STREAMS[2], STREAMS[6]):
        data = open(make_stream(workdir, name, w, h, args), "rb").read()
        assert json.loads(json.dumps(decode_with_unref(data, "port"))) == gold["unref"][name]


def _split_nals(b):
    idx, i = [], 0
    while True:
        j = b.find(b"\x00\x00\x01", i)
        if j < 0:
            break
        idx.append(j); i = j + 3
    return [b[idx[k]:(idx[k + 1] if k + 1 < len(idx) else len(b))] for k in range(len(idx))]


LOST_CASES = [("-W 3 -H 2 -n 12 -s 90292 --gop IPB --refs 5 --idr 17 --deblock 0 --wp 1", [8]),
              ("-W 3 -H 3 -n 10 -s 31 --gop IP --refs 3 --deblock 0", [5]),
              ("-W 2 -H 3 -n 30 -s 90293 --gop IPB --refs 5 --idr 9 --deblock 0 --wp 2", [24, 34, 44])]


@pytest.mark.parametrize("case", LOST_CASES, ids=["ipb_one_anchor", "ip_one_picture", "ipb_three_anchors"])
def test_lost_reference_pictures_follow_the_reference(workdir, gold, case):
    """A lost reference picture is a gap in frame_num (8.2.5.2): like the reference (edge264_headers.c:1095-1139) we insert
    non-existing frames, so the number of output frames, their order and their FrameIds must match.  Samples of pictures
    predicted from a non-existing frame are undefined in the reference (never-written buffers) and are not compared,
    except that everything output before the loss must be identical."""
    import subprocess
    from conftest import md5_frames
    from checkers import decode_bytes
    args, drop = case
    path = os.path.join(workdir, "gap_%d.264" % abs(hash(args)))
    subprocess.run([os.path.join(ROOT, "tools", "gen264"), "-o", path] + args.split(), check=True, stderr=subprocess.DEVNULL)
    nals = _split_nals(open(path, "rb").read())
    data = b"".join(n for k, n in enumerate(nals) if k not in drop)
    ref = gold["lost"][args]      # md5_before: the reference's pictures complete and output-ordered before the first loss
    ours, _ = decode_bytes(data, "port")
    assert [[f[0], f[1], f[2]] for f in ours] == ref["frames"]
    assert md5_frames(ours[:len(ref["md5_before"])]) == ref["md5_before"]


ALLOC = ctypes.CFUNCTYPE(None, ctypes.POINTER(ctypes.c_void_p), ctypes.c_uint, ctypes.POINTER(ctypes.c_void_p), ctypes.c_uint, ctypes.c_int, ctypes.c_void_p)
FREE = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p)


def decode_with_allocator(data, backend):
    """Decode with application-provided frame memory (edge264.h: Edge264AllocCb / Edge264FreeCb); returns the frames
    and the allocator traffic [(samples_size, mbs_size)], number of frees."""
    lib = load(backend)
    libc = ctypes.CDLL(None)
    libc.malloc.restype = ctypes.c_void_p; libc.malloc.argtypes = [ctypes.c_size_t]; libc.free.argtypes = [ctypes.c_void_p]
    allocs, frees, live = [], [], set()

    def on_alloc(samples, samples_size, mbs, mbs_size, err, arg):
        a = libc.malloc(samples_size + 64); b = libc.malloc(mbs_size + 64)
        samples[0] = a; mbs[0] = b
        allocs.append((samples_size, mbs_size)); live.add(a)

    def on_free(samples, mbs, arg):
        frees.append(samples); live.discard(samples)
        libc.free(samples); libc.free(mbs)

    acb, fcb = ALLOC(on_alloc), FREE(on_free)
    buf = ctypes.create_string_buffer(data, len(data) + 64)
    base = ctypes.addressof(buf); end = base + len(data)
    dec = lib.edge264_alloc(0, None, None, 0, acb, fcb, None)
    assert dec
    nal = base + 3 + (1 if data[2] == 0 else 0)
    out, f, drained = [], Edge264Frame(), False
    while True:
        sc = lib.edge264_find_start_code(nal, end, 0) if nal < end else end
        before = len(out)
        res = lib.edge264_decode_NAL(dec, nal, sc, None, None)
        if nal >= end:
            drained = True
        while lib.edge264_get_frame(dec, ctypes.byref(f), 0) == 0:
            out.append((f.FrameId, _frame_bytes(f)))
        if res == errno.ENOBUFS:
            if len(out) == before:
                break
            continue
        nal = sc + 3 if sc + 3 < end else end
        if (res not in (0, errno.ENOTSUP, errno.EBADMSG)) or drained:
            break
    d = ctypes.c_void_p(dec)
    lib.edge264_free(ctypes.byref(d))
    return out, allocs, len(frees), len(live)


def test_application_allocator_is_used_and_balanced(workdir, gold):
    name, w, h, args = STREAMS[6]
    data = open(make_stream(workdir, name, w, h, args), "rb").read()
    frames, allocs, n_free, leaked = decode_with_allocator(data, "port")
    plain, _ = decode_borrowing(data, "port", 0)
    assert [(f[0], f[1]) for f in frames] == [(f[0], f[3]) for f in plain]
    assert allocs and n_free == len(allocs) and leaked == 0, "every buffer obtained from alloc_cb must go back through free_cb"
    ref = gold["allocator"]
    assert ref["frames"] == [[f[0], hashlib.md5(f[1]).hexdigest()] for f in frames]
    assert ref["allocs"] == [list(a) for a in sorted(set(allocs))], "buffer sizes requested from the application differ from the reference's"


def sequence_changes_stream(workdir):
    import subprocess
    parts = []
    for k, a in enumerate(["-W 9 -H 7 -n 7 -s 13 --gop IPB --deblock 0", "-W 6 -H 5 -n 6 -s 14 --gop IP --refs 3 --deblock 0 --cavlc",
                           "-W 9 -H 7 -n 5 -s 15 --gop IPB --refs 4 --deblock 0", "-W 9 -H 7 -n 7 -s 13 --gop IPB --deblock 0",
                           "-W 9 -H 7 -n 4 -s 16 --gop IP --refs 1 --crop-bottom 4 --deblock 0"]):
        p = os.path.join(workdir, "seq_%d.264" % k)
        subprocess.run([os.path.join(ROOT, "tools", "gen264"), "-o", p] + a.split(), check=True, stderr=subprocess.DEVNULL)
        parts.append(open(p, "rb").read())
    return b"".join(parts)


def test_sequence_changes_follow_the_reference(workdir, gold):
    """Several coded video sequences in one stream: new sizes and crops (the reference clears its decoder), and a change of
    max_num_ref_frames alone (it does not: FrameId numbering and parameter sets continue, edge264_headers.c:2016-2024)."""
    from conftest import md5_frames
    from checkers import decode_bytes
    ref = gold["sequence"]
    ours, oc = decode_bytes(sequence_changes_stream(workdir), "port")
    assert [[f[0], f[1], f[2]] for f in ours] == ref["frames"]
    assert md5_frames(ours) == ref["md5"] and oc == ref["codes"]
