"""Multi-GPU ``train``: one process per GPU under torchrun, gradients summed over NVLink peer memory.

An N-GPU run is the same optimisation as a one-GPU run:

* ``--batch_size`` stays the global batch.  Every rank holds the whole training set on its device, draws the same
  per-epoch order from ``--tseed`` and trains on its contiguous slice of each step (``rank_slice``).
* Rank r's loss is ``sum_{i in slice} w_{y_i} l_i / W`` (``slice_loss``), W = the sum of the class weights over the whole
  step, which every rank knows because every rank has the step's labels.  The rank-order sum of the ranks' gradients
  is then the gradient of the reference's weighted-mean ``CrossEntropyLoss`` on the global batch.
* ``GradientExchange`` sums the gradients with ``dsp_comm_allreduce_f32`` (csrc/comm.cu): the fp32 sum in rank order,
  the same bits on every rank, so ``clip_grad_norm_`` and the optimizer step compute the same values everywhere and
  the replicas never drift apart.  A rank whose slice is empty (the last short step of an epoch) contributes zeros.
* Dropout masks (torch's CUDA generator) and the Philox initial states (the module's ``seed``) differ per rank, so
  the slices do not share mask and state patterns; rank 0 keeps the seeds of a one-GPU run.
* Validation batches are cut into contiguous shards, one per rank; the per-batch losses and correct counts are
  gathered, so every rank sees the same accuracy, takes the same checkpoint and early-stop decisions and stops at
  the same epoch.  Rank 0 alone writes checkpoints (the reference's names) and log lines.

The control plane (a few small ``all_gather_object`` calls) is the one ``call_freq`` uses under torchrun
(``freq_dist.join_torchrun`` / ``TorchGroup``): NCCL with a GPU per rank, gloo for ranks that share a GPU.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import time

import numpy as np
import torch
import torch.nn.functional as F

from . import _native
from . import freq_dist as fd


def rank_slice(step_len, rank, world):
    """The contiguous part of a step's ``step_len`` indices that ``rank`` trains on, as a ``slice``.  The slices of
    ranks 0..world-1 cover every index once, in order; a slice may be empty when the step has fewer sites than ranks."""
    return slice(step_len * rank // world, step_len * (rank + 1) // world)


def slice_loss(logits, y, weight, step_labels):
    """This rank's share of the weighted-mean cross entropy of a global step: ``sum w_y * l / W`` over the slice, with
    W the class-weight sum over all ``step_labels`` of the step."""
    return F.cross_entropy(logits, y, weight=weight, reduction="sum") / weight[step_labels].sum()


def window_bytes(n_elements, world):
    """Window size ``dsp_comm_allreduce_f32`` needs for ``n_elements`` floats: world slots of the 16-byte aligned
    per-rank range."""
    chunk = ((n_elements + world - 1) // world + 3) & ~3
    return max(4096, 4 * world * chunk)


class GradientExchange:
    """Deterministic in-place gradient all-reduce across the ranks of a torchrun job (``dsp_comm_allreduce_f32``).

    ``n_elements`` is the total size of the gradients it will sum (every rank passes the same value);
    ``all_gather_object`` is the control plane, e.g. ``torch.distributed.all_gather_object`` wrapped as in
    ``freq_dist.TorchGroup``.  Construction is collective."""

    def __init__(self, rank, world, device, n_elements, all_gather_object):
        if not torch.cuda.is_available():
            raise RuntimeError("the gradient all-reduce needs a CUDA device; there is no CPU path")
        self.rank, self.world = int(rank), int(world)
        self.dev = torch.device("cuda", device)
        self.n_elements = int(n_elements)
        sizes = all_gather_object(self.n_elements)
        if len(set(sizes)) != 1:
            raise ValueError("the ranks' gradients differ in size: %s" % sizes)
        self.L = _native.lib()
        self.h = C.c_void_p()
        self.h = fd.open_comm(self.rank, self.world, device, window_bytes(self.n_elements, self.world), all_gather_object)

    def allreduce_(self, params):
        """Replace ``p.grad`` of every tensor in ``params`` (e.g. ``model.parameters()``, in the same order on every rank)
        by its float32 sum over the ranks in rank order, on torch's current stream; returns when the sums are in place.
        A ``None`` grad counts as zeros and receives the sum in a new tensor.  Collective: every rank calls it."""
        params = list(params)
        grads = []
        for p in params:
            if p.grad is None:
                p.grad = torch.zeros_like(p)
            g = p.grad
            if g.dtype != torch.float32 or not g.is_contiguous() or g.device != self.dev:
                raise ValueError("allreduce_ needs contiguous float32 gradients on %s" % self.dev)
            grads.append(g)
        if sum(g.numel() for g in grads) != self.n_elements:
            raise ValueError("allreduce_: %d gradient elements, the exchange was created for %d"
                             % (sum(g.numel() for g in grads), self.n_elements))
        n = len(grads)
        ptrs = (C.c_void_p * max(n, 1))(*[g.data_ptr() for g in grads])
        numel = (C.c_int64 * max(n, 1))(*[g.numel() for g in grads])
        with torch.cuda.device(self.dev):
            stream = torch.cuda.current_stream(self.dev).cuda_stream
            _native.check(self.L.dsp_comm_allreduce_f32(self.h, ptrs, numel, n, stream), "dsp_comm_allreduce_f32")

    def close(self):
        if self.h:
            self.L.dsp_comm_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def param_digest(model):
    """SHA-256 of the names and bytes of ``model``'s ``state_dict``."""
    h = hashlib.sha256()
    for k, v in model.state_dict().items():
        h.update(k.encode())
        h.update(v.detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def check_replicas(model, all_gather_object):
    """Fail on every rank unless every rank holds the same parameters (all ranks build the model under the same
    ``--tseed`` and ``--init_model``; nothing is broadcast)."""
    digests = all_gather_object(param_digest(model))
    bad = [r for r, d in enumerate(digests) if d != digests[0]]
    if bad:
        raise RuntimeError("the model's parameters on rank(s) %s differ from rank 0's: every rank must build the model "
                           "under the same --tseed and --init_model" % bad)


def train_step(model, params, data, idx, weight, rank, world, exchange, optimizer, keys):
    """One global step on this rank's slice of ``idx``: forward + backward of ``slice_loss``, all-reduce, clip, optimizer
    step.  Returns this rank's share of the step's loss (a device scalar; the global loss is the sum over ranks)."""
    y_step = data["labels"].index_select(0, idx)
    sl = rank_slice(idx.shape[0], rank, world)
    optimizer.zero_grad()
    if sl.stop > sl.start:
        x = [data[k].index_select(0, idx[sl]) for k in keys]
        logits, _ = model(*x)
        loss = slice_loss(logits, y_step[sl], weight, y_step)
        loss.backward()
        loss = loss.detach()
    else:
        loss = torch.zeros((), device=idx.device)
    exchange.allreduce_(params)
    torch.nn.utils.clip_grad_norm_(params, 0.5)
    optimizer.step()
    return loss


def evaluate_sharded(model, data, criterion, batch_size, grp):
    """``train.evaluate`` with the validation batches cut into contiguous shards, one per rank: (mean of the per-batch
    losses, accuracy), the same on every rank."""
    from .train import KEYS
    model.eval()
    n = data["labels"].shape[0]
    nb = (n + batch_size - 1) // batch_size
    losses, correct = [], 0
    with torch.no_grad():
        for b in range(nb)[rank_slice(nb, grp.rank, grp.world)]:
            s = b * batch_size
            x = [data[k][s:s + batch_size] for k in KEYS]
            y = data["labels"][s:s + batch_size]
            logits, probs = model(*x)
            losses.append(criterion(logits, y).item())
            correct += int((torch.max(probs, 1)[1] == y).sum().item())
    model.train()
    parts = grp.all_gather_object((losses, correct))
    return float(np.mean([l for p in parts for l in p[0]])), sum(p[1] for p in parts) / n


def train_distributed(args, log=print):
    """``train.train`` across the ranks of a torchrun job (see the module docstring)."""
    from . import train as tr
    device = fd.join_torchrun("train")
    grp = fd.TorchGroup()
    rank, world = grp.rank, grp.world
    say = log if rank == 0 else (lambda *a, **k: None)
    t0 = time.time()
    dev = torch.device("cuda", device)
    torch.manual_seed(args.tseed)
    torch.cuda.manual_seed(args.tseed + rank)
    trs = tr.to_device(tr.load_feature_set(args.train_file, args.seq_len, args.signal_len), dev, "training")
    va = tr.to_device(tr.load_feature_set(args.valid_file, args.seq_len, args.signal_len), dev, "validation")
    n = trs["labels"].shape[0]
    model_dir = args.model_dir
    if rank == 0:
        os.makedirs(model_dir, exist_ok=True)
    model = tr.build_model(args, dev, seed=rank)
    check_replicas(model, grp.all_gather_object)
    weight = torch.tensor([1.0, args.pos_weight], device=dev)
    criterion = torch.nn.CrossEntropyLoss(weight=weight)
    params = list(model.parameters())
    exchange = GradientExchange(rank, world, device, sum(p.numel() for p in params), grp.all_gather_object)
    optimizer = tr.make_optimizer(args.optim_type, params, args.lr)
    scheduler = torch.optim.lr_scheduler.StepLR(optimizer, step_size=2, gamma=0.1)
    orders = tr.epoch_orders(n, args.tseed, args.max_epoch_num)
    steps = (n + args.batch_size - 1) // args.batch_size
    best, best_epoch, saved, epochs = 0.0, 0, [], 0
    say("[train] %d ranks; %d training / %d validation sites, %d steps per epoch of %d sites"
        % (world, n, va["labels"].shape[0], steps, args.batch_size))
    model.train()
    try:
        for epoch in range(args.max_epoch_num):
            best_this_epoch, no_best_model, tlosses = 0.0, True, []
            order = orders[epoch].to(dev)
            te = time.time()
            for i in range(steps):
                idx = order[i * args.batch_size:(i + 1) * args.batch_size]
                tlosses.append(train_step(model, params, trs, idx, weight, rank, world, exchange, optimizer, tr.KEYS))
                if (i + 1) % args.step_interval == 0 or i == steps - 1:
                    vloss, vacc = evaluate_sharded(model, va, criterion, args.batch_size, grp)
                    tloss = sum(grp.all_gather_object(float(torch.stack(tlosses).sum()))) / len(tlosses)
                    if vacc > best_this_epoch:
                        best_this_epoch = vacc
                        if best_this_epoch > best - 0.0002:
                            path = os.path.join(model_dir, tr.ckpt_name(args.model_type, args.seq_len, args.signal_len, epoch + 1))
                            if rank == 0:
                                torch.save(model.state_dict(), path)
                            if path not in saved:
                                saved.append(path)
                            if best_this_epoch > best:
                                best, best_epoch = best_this_epoch, epoch + 1
                            no_best_model = False
                    say("epoch [%d/%d], step [%d/%d], train loss %.4f, valid loss %.4f, valid acc %.4f, best %.4f (epoch %d)"
                        % (epoch + 1, args.max_epoch_num, i + 1, steps, tloss, vloss, vacc, best, best_epoch))
                    tlosses = []
            epochs = epoch + 1
            say("[train] epoch %d: %.1f s" % (epoch + 1, time.time() - te))
            scheduler.step()
            if no_best_model and epoch >= args.min_epoch_num - 1:
                say("[train] early stop: no better validation accuracy in epoch %d" % (epoch + 1))
                break
    finally:
        exchange.close()
    grp.barrier()                       # rank 0's checkpoints are on disk before any rank returns
    say("[train] best validation accuracy %.4f at epoch %d; %.1f s" % (best, best_epoch, time.time() - t0))
    return {"best_accuracy": best, "best_epoch": best_epoch, "checkpoints": saved, "epochs": epochs, "rank": rank,
            "world": world}
