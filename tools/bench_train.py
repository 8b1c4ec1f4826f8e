"""Training throughput of ModelBiLSTM on one GPU: the fp32 training kernels against torch/cuDNN.

One step = forward + CrossEntropy backward + clip_grad_norm_(0.5) + Adam step on a device-resident batch, as
``train.py`` runs it.  Per batch size the two arms alternate (``--rounds`` times each), each arm warms up and then
runs a timed window of ``--seconds`` ended by a device sync; CUDA events split every step into forward (through
the loss), backward, optimizer.  The torch arm is the reference's dataflow (``models.py:178-240``) on the same
module's ``nn.LSTM`` / ``nn.Linear`` containers -- cuDNN LSTMs, dropout in the reference's places.

FLOP per site are computed from the shapes: forward = the LSTM and dense contractions (2 FLOP per multiply-add),
backward = twice that (input and weight gradients), optimizer not counted.

    python tools/bench_train.py --out profiles/r03_train_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from deepsignal_plant_b200.models import ModelBiLSTM  # noqa: E402
from deepsignal_plant_b200.train import make_optimizer  # noqa: E402


def forward_flop_per_site(m):
    T, H = m.seq_len, m.hidden_size

    def lstm(K, h, layers):
        f = 0
        for l in range(layers):
            f += 2 * T * 2 * 4 * h * ((K if l == 0 else 2 * h) + h)
        return f
    f = 0
    if m.module != "signal_bilstm":
        hs = m.nhid_seq
        f += lstm((m.embedding_size if m.is_base else 0) + m.sigfea_num, hs, m.num_layers2) + 2 * T * 2 * hs * hs
    if m.module != "seq_bilstm":
        hs = m.nhid_signal
        f += lstm(m.signal_len, hs, m.num_layers2) + 2 * T * 2 * hs * hs
    f += lstm(H, H, m.num_layers1)
    return f + 2 * 2 * H * H + 2 * H * m.num_classes


def torch_forward(m, kmer, means, stds, lens, signals, p):
    """models.py:178-240 on the module's own nn containers (cuDNN), train-mode dropout."""
    T, H = m.seq_len, m.hidden_size
    parts = []
    if m.module != "signal_bilstm":
        n = kmer.shape[0]
        x = torch.cat((m.embed(kmer.long()), means.reshape(n, T, 1), stds.reshape(n, T, 1), lens.reshape(n, T, 1)), 2)
        h = torch.randn(m.num_layers2 * 2, n, m.nhid_seq, device=x.device)
        x, _ = m.lstm_seq(x, (h, torch.randn_like(h)))
        parts.append(F.relu(m.fc_seq(x)))
    if m.module != "seq_bilstm":
        n = signals.shape[0]
        h = torch.randn(m.num_layers2 * 2, n, m.nhid_signal, device=signals.device)
        x, _ = m.lstm_signal(signals, (h, torch.randn_like(h)))
        parts.append(F.relu(m.fc_signal(x)))
    x = torch.cat(parts, 2) if len(parts) > 1 else parts[0]
    h = torch.randn(m.num_layers1 * 2, x.shape[0], H, device=x.device)
    x, _ = m.lstm_comb(x, (h, torch.randn_like(h)))
    x = torch.cat((x[:, -1, :H], x[:, 0, H:]), 1)
    x = F.dropout(x, p, True)
    x = F.relu(F.dropout(m.fc1(x), p, True))
    return m.fc2(x)


def run_arm(arm, batch, seconds, warmup, p, dev, log, optim="Adam"):
    torch.manual_seed(1234)
    m = ModelBiLSTM(dropout_rate=p, trainable=True).cuda(dev).train()
    n = batch
    g = torch.Generator(device=dev).manual_seed(7)
    x = [torch.randint(0, 4, (n, 13), device=dev, generator=g).float(), torch.randn(n, 13, device=dev, generator=g),
         torch.rand(n, 13, device=dev, generator=g), torch.randint(3, 40, (n, 13), device=dev, generator=g).float(),
         torch.randn(n, 13, 16, device=dev, generator=g)]
    y = torch.randint(0, 2, (n,), device=dev, generator=g)
    crit = torch.nn.CrossEntropyLoss()
    opt = make_optimizer(optim, m.parameters(), 1e-3)
    fwd = (lambda: m(*x)[0]) if arm == "b200_kernels" else (lambda: torch_forward(m, *x, p))

    def step(ev=None):
        if ev: ev[0].record()
        loss = crit(fwd(), y)
        if ev: ev[1].record()
        opt.zero_grad()
        loss.backward()
        if ev: ev[2].record()
        torch.nn.utils.clip_grad_norm_(m.parameters(), 0.5)
        opt.step()
        if ev: ev[3].record()
        return loss
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    evs, steps = [], 0
    t0 = time.perf_counter()
    while True:
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        step(ev)
        evs.append(ev)
        steps += 1
        if steps % 4 == 0:
            torch.cuda.synchronize()
            if time.perf_counter() - t0 >= seconds:
                break
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    split = [sum(e[i].elapsed_time(e[i + 1]) for e in evs) / 1e3 for i in range(3)]
    flop = 3 * forward_flop_per_site(m)
    r = {"arm": arm, "optim": optim, "batch": batch, "steps": steps, "seconds": wall, "sites_per_s": steps * n / wall,
         "forward_s": split[0], "backward_s": split[1], "optimizer_s": split[2],
         "flop_per_site": flop, "achieved_tflops": steps * n * flop / wall / 1e12}
    log("%-12s %-6s batch %5d: %6d steps in %.2f s = %9.0f sites/s, %.2f TFLOP/s; fwd %.1f%% bwd %.1f%% opt %.1f%%" % (
        arm, optim, batch, steps, wall, r["sites_per_s"], r["achieved_tflops"], 100 * split[0] / sum(split),
        100 * split[1] / sum(split), 100 * split[2] / sum(split)))
    del m, opt
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[512, 8192])
    ap.add_argument("--seconds", type=float, default=6.0)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--dropout_rate", type=float, default=0.5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train needs a GPU")
    dev = torch.device("cuda:0")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi query failed: %s" % e
    log("card: %s | %s" % (torch.cuda.get_device_name(dev), q))
    res = []
    for b in a.batches:
        for _ in range(a.rounds):
            for arm in ("b200_kernels", "torch_cudnn"):
                res.append(run_arm(arm, b, a.seconds, a.warmup, a.dropout_rate, dev, log))
    summary = {}
    for b in a.batches:
        for arm in ("b200_kernels", "torch_cudnn"):
            rs = [r for r in res if r["batch"] == b and r["arm"] == arm]
            summary["%s_b%d_sites_per_s" % (arm, b)] = max(r["sites_per_s"] for r in rs)
    log(json.dumps(summary))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"card": torch.cuda.get_device_name(dev), "nvidia_smi": q, "model": "both_bilstm 13x16 hidden 256, "
                       "3+1 layers, dropout %.1f, Adam" % a.dropout_rate, "runs": res, "summary": summary}, f, indent=1)
        with open(os.path.splitext(a.out)[0] + ".log", "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
