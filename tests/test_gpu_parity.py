"""GPU parity proper: the sm_100a kernels behind the edge264 C API against the oracle and the golden digests of the
reference's output — bit-exact, every frame."""
import json, os, subprocess
import pytest
from conftest import ROOT, STREAMS, DPB_STREAMS, make_stream, md5_frames
from checkers import decode_bytes

pytestmark = pytest.mark.gpu
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "streams.json")))


# the decoded-picture-buffer streams too: slices of different types in one picture put intra and inter macroblocks side by
# side in every proportion (an intra-heavy P picture once took the intra-picture wavefront past a neighbour still in work)
ALL_STREAMS = STREAMS + DPB_STREAMS


@pytest.mark.parametrize("name,w,h,args", ALL_STREAMS, ids=[s[0] for s in ALL_STREAMS])
def test_gpu_matches_oracle_and_golden(workdir, name, w, h, args):
    data = open(make_stream(workdir, name, w, h, args), "rb").read()
    gpu, codes = decode_bytes(data, "gpu")
    assert md5_frames(gpu) == GOLD[name]["md5"]
    port, pcodes = decode_bytes(data, "port")
    assert md5_frames(gpu) == md5_frames(port) and codes == pcodes
    assert [f[0] for f in gpu] == [f[0] for f in port]


FULL = [
    ("1080p_intra", 120, 68, "-n 4 -s 31 --gop I --deblock 0 --t8x8 50 --density 40"),
    ("1080p_ipb", 120, 68, "-n 13 -s 32 --gop IPB --deblock 0 --t8x8 50 --density 52 --wp 2"),
    ("2160p_scaling", 240, 135, "-n 7 -s 33 --gop IPB --deblock 0 --t8x8 70 --scaling 3 --density 40 --qp 30"),
    # BASELINE configs[4]: 7680x4320 level 6.2, B slices with explicit / implicit weighted bi-prediction, every edge filtered
    ("4320p_wp_explicit", 480, 270, "-n 4 -s 34 --gop IPB --deblock 0 --wp 1 --density 60 --skip-pct 0 --refs 2"),
    ("4320p_wp_implicit", 480, 270, "-n 4 -s 35 --gop IPB --deblock 0 --wp 2 --density 60 --skip-pct 5 --temporal"),
]


@pytest.mark.parametrize("name,w,h,args", FULL, ids=[s[0] for s in FULL])
def test_full_size_against_reference(workdir, name, w, h, args):
    """BASELINE.json sizes: compared with the reference decoder's frame count, last return code and output signature
    (tests/golden/full_size.json, from the same tools/e264_decode.c over the compiled reference; the oracle port is too
    slow here)."""
    path = make_stream(workdir, name, w, h, args)
    ref = json.load(open(os.path.join(ROOT, "tests", "golden", "full_size.json")))[name]
    gpu = subprocess.run([os.path.join(ROOT, "tools", "b200_decode"), path, "-q"], capture_output=True, text=True, timeout=600).stdout.strip().splitlines()[-1]
    assert ref == gpu and ref.startswith("frames")


def test_replay_reproduces_decode(workdir):
    """Size-independent property: re-running the kept device records (bench.py's kernel-only path)
    leaves every frame slot with exactly the pixels the live decode produced."""
    import ctypes
    os.environ["E264B_KEEP"] = "1"
    try:
        path = make_stream(workdir, "replay", 20, 12, "-n 9 -s 41 --gop IPB --deblock 0 --wp 1")
        bench = ctypes.CDLL(os.path.join(ROOT, "tools", "libe264bench.so"))
        core = ctypes.CDLL(os.path.join(ROOT, "edge264_b200", "libedge264_b200.so"))
        bench.e264bench_run.restype = ctypes.c_double
        core.e264b_of_decoder.restype = ctypes.c_void_p; core.e264b_of_decoder.argtypes = [ctypes.c_void_p]
        core.e264b_slot_hash.restype = ctypes.c_uint64; core.e264b_slot_hash.argtypes = [ctypes.c_void_p, ctypes.c_int]
        data = open(path, "rb").read()
        bufs = (ctypes.c_char_p * 1)(data); sizes = (ctypes.c_size_t * 1)(len(data))
        frames = (ctypes.c_long * 1)(); sums = (ctypes.c_uint64 * 1)(); decs = (ctypes.c_void_p * 1)()
        bench.e264bench_run(bufs, sizes, 1, 1, 1, frames, sums, decs)
        dev = core.e264b_of_decoder(decs[0])
        before = [core.e264b_slot_hash(dev, s) for s in range(4)]
        import bench as benchmod      # (the local name `bench` is the driver library)
        devs = (ctypes.c_void_p * 1)(dev); st = benchmod.ReplayStats()
        core.e264b_replay.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(benchmod.ReplayStats)]
        assert core.e264b_replay(devs, 1, 2, 1, ctypes.byref(st)) == 0
        assert [core.e264b_slot_hash(dev, s) for s in range(4)] == before
        # per picture: inter (if any), intra (if any), deblock -> 2..3 launches here, replayed twice
        assert 2 * 2 * frames[0] <= st.launches <= 2 * 3 * frames[0] and core.e264b_error_flag(dev) == 0
        assert sum(st.kernel_launches) == st.launches and st.kernel_ms[3] > 0 and st.kernel_ms[0] == 0 and st.kernel_ms[4] == 0
        bench.e264bench_free(decs, 1)
    finally:
        os.environ["E264B_KEEP"] = "0"
