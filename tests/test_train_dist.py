"""Multi-GPU training (train_dist.py + dsp_comm_allreduce_f32 in csrc/comm.cu).

CPU (``-m "not gpu"``): how a step is cut over the ranks, the global-weight normalisation of the per-rank loss, and the
argument checks of the all-reduce entry that need no device.
GPU (``-m gpu``): 2-4 ranks that SHARE cuda:0 (CUDA IPC works between processes on one device; the control plane runs on
gloo): the all-reduce bit for bit against numpy's float32 sum in rank order, gradient parity of a split batch against
the float64 oracle of the whole batch, no drift of the replicas over Adam steps, the start-up check, and the ``train``
command under torchrun.  With two GPUs the all-reduce and ``train`` also run over real NVLink."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from deepsignal_plant_b200 import _native, cli
from deepsignal_plant_b200 import train as tr
from deepsignal_plant_b200 import train_dist as td

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKER = os.path.join(ROOT, "tests", "train_dist_worker.py")
TWO_GPUS = torch.cuda.is_available() and torch.cuda.device_count() >= 2


def _run_ranks(world, args, timeout=900, env_extra=None, module=None):
    port = 29400 + (os.getpid() * 11 + world * 17 + len(args)) % 2000
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(port)]
    cmd += (["-m", module] if module else [WORKER]) + [str(a) for a in args]
    env = dict(os.environ)
    env.update(env_extra or {})
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-5000:]
    return r.stdout


def _verdict(out):
    return json.loads([l for l in out.splitlines() if l.startswith("{")][-1])


# ---- CPU -------------------------------------------------------------------------------------------------------
def test_rank_slices_cover_every_index_once_in_order():
    for world in range(1, 9):
        for batch in (1, 3, 7, 8, 37, 512, 513):
            for n in (1, 5, 100, 513, 1024, 4097):
                steps = (n + batch - 1) // batch
                for i in range(steps):
                    idx = list(range(i * batch, min(n, (i + 1) * batch)))           # the last step may be short
                    parts = [idx[td.rank_slice(len(idx), r, world)] for r in range(world)]
                    assert sum(parts, []) == idx, (world, batch, n, i)
                    sizes = [len(p) for p in parts]
                    assert max(sizes) - min(sizes) <= 1
                    if len(idx) < world:
                        assert 0 in sizes


def test_global_weight_normalisation_sums_to_the_weighted_mean_gradient():
    torch.manual_seed(0)
    n, d = 53, 6
    x = torch.randn(n, d, dtype=torch.float64)
    y = (torch.rand(n) < 0.2).long()                                               # unbalanced labels
    weight = torch.tensor([1.0, 3.7], dtype=torch.float64)
    w0 = torch.randn(d, 2, dtype=torch.float64)
    full = w0.clone().requires_grad_()
    torch.nn.CrossEntropyLoss(weight=weight)(x @ full, y).backward()
    for world in (1, 2, 3, 4, 8, 60):
        acc = torch.zeros_like(w0)
        total = 0.0
        for r in range(world):
            sl = td.rank_slice(n, r, world)
            part = w0.clone().requires_grad_()
            loss = td.slice_loss(x[sl] @ part, y[sl], weight, y)
            loss.backward()
            acc += part.grad
            total += float(loss.detach())
        assert torch.allclose(acc, full.grad, rtol=1e-12, atol=1e-15), world
        assert abs(total - float(torch.nn.CrossEntropyLoss(weight=weight)(x @ w0, y))) < 1e-12


def test_window_size_holds_every_rank_slot():
    for e in (0, 1, 7, 4694082, 71006):
        for world in range(1, 9):
            chunk = ((e + world - 1) // world + 3) & ~3
            assert chunk % 4 == 0 and chunk * world >= e
            assert td.window_bytes(e, world) >= 4 * world * chunk


def test_allreduce_entry_rejects_bad_arguments_without_a_device():
    L = _native.lib()
    buf = (C.c_float * 8)()
    one = (C.c_void_p * 1)(C.addressof(buf))
    cases_ = [("n_bufs", one, (C.c_int64 * 1)(8), -1),
              ("numel", one, (C.c_int64 * 1)(-3), 1),
              ("numel", one, (C.c_int64 * 1)(1 << 62), 1),
              ("null buffer", None, None, 2),
              ("bufs[0] is null", (C.c_void_p * 1)(None), (C.c_int64 * 1)(4), 1),
              ("null communicator", one, (C.c_int64 * 1)(8), 1)]
    for what, ptrs, numel, n in cases_:
        rc = L.dsp_comm_allreduce_f32(None, ptrs, numel, n, None)
        assert rc == 1, what
        assert what.encode() in L.dsp_last_error(), (what, L.dsp_last_error())


def test_train_dispatches_to_the_distributed_loop_only_under_torchrun(monkeypatch):
    called = []
    monkeypatch.setattr(td, "train_distributed", lambda args, log=print: called.append(args) or {"rank": 0})
    args = cli.build_parser().parse_args(["train", "--train_file", "t", "--valid_file", "v", "--model_dir", "m"])
    monkeypatch.setenv("WORLD_SIZE", "2")
    assert tr.train(args) == {"rank": 0} and called == [args]
    monkeypatch.setenv("WORLD_SIZE", "1")
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU path"):
            tr.train(args)
        assert len(called) == 1


# ---- GPU: ranks sharing cuda:0 -------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 4])
def test_allreduce_is_the_rank_order_float32_sum_bit_for_bit(world):
    v = _verdict(_run_ranks(world, ["allreduce"]))
    # a sum of two floats is correctly rounded in either order; from three ranks on the order shows in the bits
    assert v["ok"] and (world < 3 or v["order_matters"]), v
    for e in v["ranks"]:
        assert len(set(e["digests"])) == 1                                         # a second call gives the same bits
        assert e["errors"]["oversized"][0] == 4 and "windows of" in e["errors"]["oversized"][1]
        assert e["errors"]["negative"][0] == 1 and e["errors"]["null_buffer"][0] == 1
        assert "created for" in e["errors"]["wrong_total"]


@pytest.mark.gpu
@pytest.mark.parametrize("dropout", [0.0, 0.5])
@pytest.mark.parametrize("world,hidden", [(2, 256), (3, 32), (4, 32)])
def test_split_batch_gradients_match_the_whole_batch_oracle(world, hidden, dropout):
    v = _verdict(_run_ranks(world, ["parity", "--hidden", hidden, "--sites", 37, "--dropout", dropout]))
    print("split-batch parity world %d H=%d p=%.1f: worst logit err %.2e, worst grad err %.2e x max|g|"
          % (world, hidden, dropout, max(e["logit_err"] for e in v["ranks"]), max(e["grad_err"] for e in v["ranks"])))
    assert v["ok"], v


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_replicas_stay_bit_identical_over_adam_steps(world):
    v = _verdict(_run_ranks(world, ["drift"]))
    assert v["ok"], v


@pytest.mark.gpu
def test_startup_check_fails_on_every_rank_when_one_differs():
    v = _verdict(_run_ranks(2, ["perturb"]))
    assert v["ok"], v


def _train_pair(tmp_path):
    from test_train import write_pair
    _, tr_bin, _ = write_pair(tmp_path, 8193, seed=31, name="train")              # 17 steps of 512: the last has one site
    _, va_bin, va_labels = write_pair(tmp_path, 1024, seed=32, name="valid")
    return tr_bin, va_bin, va_labels


def _check_checkpoints_load(mdir, res, va_bin, va_labels, tmp_path):
    names = sorted(os.listdir(mdir))
    assert names == sorted(os.path.basename(p) for p in res["checkpoints"]), names
    assert all(n.startswith("both_bilstm.b13_s16_epoch") and n.endswith(".ckpt") for n in names)
    best = os.path.join(mdir, tr.ckpt_name("both_bilstm", 13, 16, res["best_epoch"]))
    out = tmp_path / "calls.tsv"
    assert cli.main(["call_mods", "-i", va_bin, "-m", best, "-o", str(out)]) == 0
    called = np.array([int(line.split("\t")[8]) for line in open(out)])
    assert len(called) == len(va_labels) and float((called == va_labels).mean()) >= 0.9


@pytest.mark.gpu
def test_train_command_two_ranks_sharing_one_gpu(tmp_path):
    tr_bin, va_bin, va_labels = _train_pair(tmp_path)
    mdir = tmp_path / "models"
    v = _verdict(_run_ranks(2, ["train", "--train_file", tr_bin, "--valid_file", va_bin, "--model_dir", mdir,
                                "--max_epoch_num", 4, "--min_epoch_num", 2, "--step_interval", 8]))
    print("train, 2 ranks on one GPU:", v["ranks"][0])
    assert v["ok"], v                                            # same epochs, best epoch and checkpoints on both ranks
    assert v["ranks"][0]["best_accuracy"] >= 0.9
    _check_checkpoints_load(mdir, v["ranks"][0], va_bin, va_labels, tmp_path)


# ---- GPU: two physical GPUs (NVLink) -------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.skipif(not TWO_GPUS, reason="needs two GPUs")
def test_allreduce_over_nvlink_is_bit_exact():
    v = _verdict(_run_ranks(2, ["allreduce"]))
    assert v["ok"], v


@pytest.mark.gpu
@pytest.mark.skipif(not TWO_GPUS, reason="needs two GPUs")
def test_train_command_two_gpus(tmp_path):
    tr_bin, va_bin, va_labels = _train_pair(tmp_path)
    mdir = tmp_path / "models"
    out = _run_ranks(2, ["train", "--train_file", tr_bin, "--valid_file", va_bin, "--model_dir", mdir, "--max_epoch_num", 4,
                         "--min_epoch_num", 2, "--step_interval", 8], module="deepsignal_plant_b200")
    assert "[train] 2 ranks" in out and out.count("[train] best validation accuracy") == 1, out
    names = sorted(os.listdir(mdir))
    assert names and all(n.startswith("both_bilstm.b13_s16_epoch") and n.endswith(".ckpt") for n in names)
