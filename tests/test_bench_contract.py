"""bench.py contract pieces: the reference arm prints one JSON line with the agreed keys; FLOP bookkeeping
matches SURVEY.md section 8d; --dump-outputs stays within its size limit and, on the GPU, writes what the last
timed step returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "sites/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["metric"].startswith("classified sites/sec") and d["steps"] == 1 and d["scaling"] == "weak"
    # the unmodified reference from oracle/_ref when it is built (kind "reference"), else the torch-operator port
    sys.path.insert(0, ROOT)
    from oracle import ref_import
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_import.available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "sites/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_flop_bookkeeping_matches_survey():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.flops_per_site("both_bilstm", 13, 16)[0] == 118447104
    assert bench.flops_per_site("seq_bilstm", 13, 16)[0] == 126727168
    assert bench.flops_per_site("signal_bilstm", 13, 16)[0] == 127206400
    assert bench.flops_per_site("both_bilstm", 17, 20)[0] == 154950656


def test_bench_refuses_to_run_without_gpu():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                       timeout=300, cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode != 0 and "needs a GPU" in (r.stderr + r.stdout)


def test_traffic_capture_is_tied_to_the_kernel_source():
    # roofline.traffic comes from an ncu capture; bench.py must refuse to quote it for another version of the kernels
    sys.path.insert(0, ROOT)
    import hashlib
    import bench
    t, detail = bench.traffic_of_dominant_kernel(65536)
    d = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
    sha = hashlib.sha256(open(os.path.join(ROOT, "deepsignal_plant_b200", "csrc", "kernels_tc.cu"), "rb").read()).hexdigest()
    if d.get("kernels_tc_sha256") == sha:
        assert t == d["dram_bytes_per_site"] * 65536
    else:
        assert t is None and "re-capture" in detail["reason"]


def test_command_line_object_reports_instead_of_raising():
    # bench.py's `cli` object runs tools/bench_cli.py --binary in a subprocess: with the device stubbed out it yields the
    # numbers of the host pipeline; without a GPU the real command fails and the object says so -- the bench line never
    # depends on it
    sys.path.insert(0, ROOT)
    import bench
    small = ["--block-sites", "4096"]
    d = bench.command_line_run(9000, extra=["--host-only"] + small)
    assert "unavailable" not in d and d["sites"] == 8192 == d["lines_written"] and d["value"] > 0 and d["unit"] == "sites/s"
    import torch
    if not torch.cuda.is_available():
        d = bench.command_line_run(9000, extra=small)
        assert set(d) == {"unavailable"} and "CUDA" in d["unavailable"]


def test_dump_outputs_needs_the_device_forward(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--dump-outputs", str(tmp_path / "d")], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and not os.path.exists(tmp_path / "d")


def test_dump_outputs_samples_rows_within_the_size_limit(tmp_path):
    sys.path.insert(0, ROOT)
    import torch
    import bench
    arrays = [("probs", torch.arange(1000, dtype=torch.float32).reshape(500, 2)), ("labels", torch.arange(500, dtype=torch.int32))]
    bench.dump_outputs(str(tmp_path / "all"), arrays, max_bytes=500 * 12)
    assert sorted(os.listdir(tmp_path / "all")) == ["labels.npy", "probs.npy"]
    assert np.array_equal(np.load(tmp_path / "all" / "probs.npy"), arrays[0][1].numpy())
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, max_bytes=4000)
    got = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in ("rows", "probs", "labels")}
    for n in got:
        assert got[n].dtype == (np.float64 if n == "rows" else np.float32)
        assert np.array_equal(got[n], np.load(tmp_path / "b" / (n + ".npy")))          # the same seeded sample
    rows = got["rows"].astype(np.int64)
    assert len(rows) == 4000 // 20 and (np.diff(rows) > 0).all() and rows[-1] < 500
    assert sum(a.nbytes for a in got.values()) <= 4000
    assert np.array_equal(got["probs"], arrays[0][1].numpy()[rows]) and np.array_equal(got["labels"], rows)


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(tmp_path):
    # the dump must be what the last of --steps timed forwards returned: recompute that step here (same weights, same
    # input batch of the cycled pool, same Philox call count) and count the timed launches
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from deepsignal_plant_b200.models import ModelBiLSTM
    steps, warmup = 3, 3
    d = str(tmp_path / "dump")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                        "--precision", "fp16", "--no-cpu-baseline", "--no-freq", "--no-cli", "--dump-outputs", d],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    got = {n: np.load(os.path.join(d, n + ".npy")) for n in ("logits", "probs", "labels")}
    assert sorted(os.listdir(d)) == ["labels.npy", "logits.npy", "probs.npy"]

    torch.manual_seed(1234)
    model = ModelBiLSTM(13, 16, 3, 1, 2, 0, 256, 16, 4, True, True, module="both_bilstm", device=0, precision="fp16",
                        max_batch=bench.BATCH, seed=0).cuda(0).eval()
    pool = [tuple(torch.from_numpy(a).cuda(0) for a in b) for b in bench.make_pool(4, bench.BATCH, seed=0)]
    for i in range(warmup):
        model(*pool[i % 4])
    for i in range(steps - 1):
        model(*pool[i % 4])
    l0 = model.launch_count()
    logits, probs = model(*pool[(steps - 1) % 4])
    want = {"logits": logits.cpu().numpy(), "probs": probs.cpu().numpy(), "labels": model.last_labels.float().cpu().numpy()}
    for n in got:
        assert got[n].dtype == np.float32 and got[n].shape == want[n].shape and np.array_equal(got[n], want[n]), n
    assert line["steps"] == steps and line["gpu_launches"] == steps * (model.launch_count() - l0)
    assert (got["labels"] == got["probs"].argmax(1)).all()
