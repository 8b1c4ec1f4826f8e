"""One rank of the multi-rank training tests (launched by torchrun from test_train_dist.py).  Every mode gathers one
record per rank; rank 0 prints them, with the verdict of the checks that need every rank's answer, as one JSON line."""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from deepsignal_plant_b200 import _native, synthetic  # noqa: E402
from deepsignal_plant_b200 import freq_dist as fd  # noqa: E402
from deepsignal_plant_b200 import train_dist as td  # noqa: E402
from deepsignal_plant_b200.models import ModelBiLSTM  # noqa: E402

KEYS = ("kmer", "base_means", "base_stds", "base_signal_lens", "signals")
SIZES = [7, 1, 1023, 0, 333, 4099, 65536 + 5, 2]          # total 71006: not a multiple of 4, 3 or any world size here
NONE_AT = 2                                                # the last rank has no gradient for this tensor


def rank_values(r, world):
    """Rank r's gradients: mostly O(1) values with +-1e8 next to them, so that the order of summation changes the result."""
    rng = np.random.default_rng(1000 + r)
    out = []
    for i, n in enumerate(SIZES):
        v = rng.standard_normal(n).astype(np.float32)
        big = rng.random(n) < 0.3
        v[big] = np.where(rng.random(int(big.sum())) < 0.5, -1e8, 1e8).astype(np.float32) * (1 + rng.random(int(big.sum())).astype(np.float32))
        out.append(None if (r == world - 1 and i == NONE_AT) else v)
    return out


def expected_sums(world, order):
    acc = None
    for r in order:
        vals = [np.zeros(n, np.float32) if v is None else v for v, n in zip(rank_values(r, world), SIZES)]
        acc = vals if acc is None else [(a + b).astype(np.float32) for a, b in zip(acc, vals)]
    return acc


def emit(grp, mine, verdict):
    every = grp.all_gather_object(mine)
    if grp.rank == 0:
        print(json.dumps(dict(verdict(every), ranks=every)), flush=True)


def mode_allreduce(grp, device):
    world, rank = grp.world, grp.rank
    dev = torch.device("cuda", device)
    params = [torch.zeros(n, device=dev, requires_grad=True) for n in SIZES]
    ex = td.GradientExchange(rank, world, device, sum(SIZES), grp.all_gather_object)
    want = expected_sums(world, range(world))
    exact64 = [np.zeros(n, np.float64) for n in SIZES]
    for r in range(world):
        for acc, v in zip(exact64, rank_values(r, world)):
            acc += 0.0 if v is None else v.astype(np.float64)
    order_matters = any(not np.array_equal(a, b.astype(np.float32)) for a, b in zip(want, exact64))
    digests, exact = [], True
    for _ in range(2):
        for p, v in zip(params, rank_values(rank, world)):
            p.grad = None if v is None else torch.from_numpy(v).to(dev)
        ex.allreduce_(params)
        got = [p.grad.cpu().numpy() for p in params]
        exact = exact and all(np.array_equal(g.view(np.uint32), w.view(np.uint32)) for g, w in zip(got, want))
        digests.append(hashlib.sha256(b"".join(g.tobytes() for g in got)).hexdigest())
    # argument checks on a live communicator: every rank takes the same error path, nothing is launched
    L = _native.lib()
    errors = {}
    big = torch.zeros(sum(SIZES) * 2 + 4096, device=dev)
    for name, ptrs, numel in (("oversized", [big.data_ptr()], [big.numel()]),
                              ("negative", [big.data_ptr()], [-5]),
                              ("null_buffer", [None], [16])):
        rc = L.dsp_comm_allreduce_f32(ex.h, (C.c_void_p * 1)(*ptrs), (C.c_int64 * 1)(*numel), 1,
                                      torch.cuda.current_stream(dev).cuda_stream)
        errors[name] = [int(rc), L.dsp_last_error().decode()]
    try:
        ex.allreduce_(params[:-1])
        errors["wrong_total"] = "accepted"
    except ValueError as e:
        errors["wrong_total"] = str(e)
    ex.close()
    emit(grp, {"exact": bool(exact), "digests": digests, "errors": errors},
         lambda every: {"ok": all(e["exact"] for e in every) and len({d for e in every for d in e["digests"]}) == 1,
                        "order_matters": bool(order_matters)})


def build(H, p, dev, state_mode="init_hidden", seed=0):
    torch.manual_seed(1234)
    return ModelBiLSTM(13, 16, 3, 1, 2, p, H, 16, 4, True, True, module="both_bilstm", precision="fp32",
                       state_mode=state_mode, seed=seed, trainable=True).cuda(dev)


def mode_parity(grp, device, H, n, p):
    """Split one global batch over the ranks (slices of explicit initial states and dropout masks); after the
    all-reduce every rank's gradients must match the float64 oracle of the whole batch."""
    from oracle import model_oracle, train_oracle
    world, rank = grp.world, grp.rank
    dev = torch.device("cuda", device)
    model = build(H, p, dev).train()
    f = synthetic.make_features(n, 13, 16, seed=n)
    labels = np.random.default_rng(n).integers(0, 2, n)
    labels[: n // 4] = 1                                        # unbalanced with pos_weight != 1
    cfg = model_oracle.make_cfg(13, 16, 3, 1, 2, H)
    states = synthetic.make_states(cfg, n, seed=77)
    g = torch.Generator().manual_seed(5)
    masks = [None if s is None or p == 0 else (torch.rand(s, generator=g) >= p).float() / (1 - p)
             for s in model.dropout_mask_shapes(n)]
    sl = td.rank_slice(n, rank, world)
    order = iter(["seq", "signal", "comb"])
    model.init_hidden = lambda b, l, h: tuple(torch.from_numpy(x[:, sl]).contiguous().to(dev) for x in states[next(order)])
    model.draw_dropout_masks = lambda m, d: [None if x is None else x[sl].contiguous().to(d) for x in masks]
    weight = torch.tensor([1.0, 2.5], device=dev)
    y = torch.from_numpy(labels).to(dev)
    ex = td.GradientExchange(rank, world, device, sum(q.numel() for q in model.parameters()), grp.all_gather_object)
    logits, _ = model(*[torch.from_numpy(f[k][sl]).to(dev) for k in KEYS])
    td.slice_loss(logits, y[sl], weight, y).backward()
    ex.allreduce_(model.parameters())
    ex.close()
    sd = {k: v.detach().cpu().double().requires_grad_() for k, v in model.state_dict().items()}
    st = {k: (torch.from_numpy(h_), torch.from_numpy(c_)) for k, (h_, c_) in states.items()}
    want_logits = train_oracle.forward(sd, cfg, *(torch.from_numpy(f[k]) for k in KEYS), st, masks)
    torch.nn.functional.cross_entropy(want_logits, torch.from_numpy(labels), weight=weight.cpu().double()).backward()
    lerr = float((logits.detach().cpu().double() - want_logits.detach()[sl]).abs().max()) if sl.stop > sl.start else 0.0
    worst = 0.0
    for name, prm in model.named_parameters():
        w = sd[name].grad
        worst = max(worst, float((prm.grad.cpu().double() - w).abs().max()) / (float(w.abs().max()) or 1.0))
    digest = hashlib.sha256(b"".join(q.grad.cpu().numpy().tobytes() for q in model.parameters())).hexdigest()
    emit(grp, {"logit_err": lerr, "grad_err": worst, "digest": digest},
         lambda every: {"ok": all(e["logit_err"] < 1e-5 and e["grad_err"] < 1e-4 for e in every)
                        and len({e["digest"] for e in every}) == 1})


def mode_drift(grp, device, steps=10):
    """Adam with clipping and dropout 0.5 on the training step of train_dist; the last step has one site, so the
    other ranks contribute no gradient there.  The parameters must stay bit-identical on every rank."""
    world, rank = grp.world, grp.rank
    dev = torch.device("cuda", device)
    torch.cuda.manual_seed(99 + rank)
    model = build(64, 0.5, dev, state_mode="philox", seed=rank).train()
    n = 96
    f = synthetic.make_features(n, 13, 16, seed=3)
    data = {k: torch.from_numpy(f[k]).to(dev) for k in KEYS}
    data["labels"] = torch.from_numpy(np.random.default_rng(4).integers(0, 2, n)).to(dev)
    params = list(model.parameters())
    ex = td.GradientExchange(rank, world, device, sum(q.numel() for q in params), grp.all_gather_object)
    opt = torch.optim.Adam(params, lr=1e-3)
    weight = torch.tensor([1.0, 1.7], device=dev)
    losses = []
    for s in range(steps):
        idx = torch.arange(n, device=dev) if s < steps - 1 else torch.tensor([n - 1], device=dev)
        losses.append(float(td.train_step(model, params, data, idx, weight, rank, world, ex, opt, KEYS)))
    ex.close()
    ok = True
    try:
        td.check_replicas(model, grp.all_gather_object)
    except RuntimeError:
        ok = False
    emit(grp, {"digest": td.param_digest(model), "losses": losses, "replicas_agree": ok},
         lambda every: {"ok": len({e["digest"] for e in every}) == 1 and all(e["replicas_agree"] for e in every)})


def mode_perturb(grp, device):
    dev = torch.device("cuda", device)
    model = build(32, 0.0, dev)
    if grp.rank == grp.world - 1:
        with torch.no_grad():
            model.fc2.bias[0] += 1e-6
    try:
        td.check_replicas(model, grp.all_gather_object)
        msg = None
    except RuntimeError as e:
        msg = str(e)
    emit(grp, {"error": msg}, lambda every: {"ok": all(e["error"] and "differ" in e["error"] for e in every)})


def mode_train(grp, argv):
    from deepsignal_plant_b200 import cli
    from deepsignal_plant_b200 import train as tr
    res = tr.main(cli.build_parser().parse_args(["train"] + argv))
    emit(grp, res, lambda every: {"ok": len({(e["epochs"], e["best_epoch"], tuple(e["checkpoints"])) for e in every}) == 1})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("mode", choices=["allreduce", "parity", "drift", "perturb", "train"])
    ap.add_argument("--hidden", type=int, default=32)
    ap.add_argument("--sites", type=int, default=37)       # not --n: torchrun's parser would take it for one of its own
    ap.add_argument("--dropout", type=float, default=0.0)
    a, rest = ap.parse_known_args()
    dist.init_process_group("gloo")
    device = int(os.environ.get("LOCAL_RANK", "0")) % torch.cuda.device_count()
    torch.cuda.set_device(device)
    grp = fd.TorchGroup()
    if a.mode == "allreduce":
        mode_allreduce(grp, device)
    elif a.mode == "parity":
        mode_parity(grp, device, a.hidden, a.sites, a.dropout)
    elif a.mode == "drift":
        mode_drift(grp, device)
    elif a.mode == "perturb":
        mode_perturb(grp, device)
    else:
        mode_train(grp, rest)
    grp.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
