"""bench.py's reference arm needs no GPU: run it on a tiny batch and check the one-JSON-line contract
(metric/unit/value, impl, cpu_baseline, e2e) and --dump-outputs.  The reference arm's driver (tools/e264_bench.c) is
linked here against the CPU checker build of the decoder (oracle/liboracle_dec.so) in place of the compiled reference,
in a tree with bench.py's layout, so the tests need neither the reference's sources nor a GPU.  The GPU arm's dump is
checked against that stand-in on the B200."""
import json, os, subprocess, sys
import numpy as np
import pytest
from conftest import ROOT

TINY = ["--steps", "1", "--warmup", "1", "--streams", "2", "--frames", "6"]


@pytest.fixture(scope="module")
def standin(tmp_path_factory):
    root = tmp_path_factory.mktemp("standin")
    os.makedirs(root / "tools"); os.makedirs(root / "oracle" / "_ref")
    os.symlink(os.path.join(ROOT, "bench.py"), root / "bench.py")
    os.symlink(os.path.join(ROOT, "tools", "gen264"), root / "tools" / "gen264")
    subprocess.run(["gcc", "-O2", "-std=gnu11", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tools", "e264_bench.c"),
                    "-o", str(root / "oracle" / "_ref" / "libe264bench_ref.so"), os.path.join(ROOT, "oracle", "liboracle_dec.so"), "-pthread"], check=True)
    return str(root / "bench.py")


def run_bench(bench, args, workdir):
    r = subprocess.run([sys.executable, bench] + args + ["--workdir", str(workdir)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-800:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "stdout must carry exactly one line"
    return json.loads(lines[0])


def test_reference_arm_prints_one_json_line(standin, tmp_path):
    d = run_bench(standin, ["--impl", "reference"] + TINY, tmp_path)
    assert d["impl"] == "reference" and d["metric"] == "1080p_high_cabac_ipb_decode_fps" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def load_dump(path):
    files = sorted(os.listdir(path))
    assert files == ["frame_info.npy", "frames.npy"]
    assert sum(os.path.getsize(os.path.join(path, f)) for f in files) <= 64 << 20
    out = {f: np.load(os.path.join(path, f)) for f in files}
    assert out["frames.npy"].dtype == np.float32 and out["frame_info.npy"].dtype == np.float64
    return out


def test_dump_outputs_are_the_same_from_run_to_run(standin, tmp_path):
    """Same arguments, same dump, whatever the number of steps (the last timed step is dumped) and with the streams
    generated afresh or taken from the cache."""
    a = ["--impl", "reference", "--streams", "2", "--frames", "6", "--dump-outputs"]
    run_bench(standin, a + [str(tmp_path / "a"), "--steps", "1", "--warmup", "0"], tmp_path / "w1")
    run_bench(standin, a + [str(tmp_path / "b"), "--steps", "3", "--warmup", "1"], tmp_path / "w1")
    run_bench(standin, a + [str(tmp_path / "c"), "--steps", "2", "--warmup", "0"], tmp_path / "w2")
    da, db, dc = (load_dump(tmp_path / k) for k in "abc")
    info = da["frame_info.npy"]
    assert len(info) == 12 and (info[:, 3:5] == [1920, 1080]).all() and da["frames.npy"].shape[0] == 12
    for d in (db, dc):
        for k in da:
            assert np.array_equal(da[k], d[k]), k


@pytest.mark.gpu
def test_gpu_arm_dump_matches_the_oracle(standin, tmp_path):
    """The GPU arm's dump of its last timed step equals the CPU checker's on the same inputs."""
    d = run_bench(os.path.join(ROOT, "bench.py"), TINY + ["--dump-outputs", str(tmp_path / "gpu")], tmp_path / "w")
    assert d["steps"] == 1 and d["value"] > 0
    run_bench(standin, ["--impl", "reference"] + TINY + ["--dump-outputs", str(tmp_path / "cpu")], tmp_path / "w")
    gpu, cpu = load_dump(tmp_path / "gpu"), load_dump(tmp_path / "cpu")
    for k in gpu:
        assert np.array_equal(gpu[k], cpu[k]), k
