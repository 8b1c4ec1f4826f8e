"""``train``: the reference's training loop (``deepsignal_plant/train.py``, SURVEY §3.4) on the fp32
training kernels.

Loop, as the reference runs it:
* CrossEntropyLoss with class weights [1, pos_weight]; Adam / RMSprop / SGD(momentum 0.8) at ``--lr``;
  StepLR(step_size=2, gamma=0.1) stepped once per epoch; ``clip_grad_norm_(model.parameters(), 0.5)``.
* Every ``step_interval`` steps and at the last step of an epoch the model is validated under
  ``eval()`` (the inference path).  When the validation accuracy beats the best of this epoch and comes
  within 0.0002 of the best so far, the bare ``state_dict`` is saved as
  ``{model_type}.b{seq_len}_s{signal_len}_epoch{n}.ckpt`` (n counts from 1).
* Stopping rule: after an epoch that saved no checkpoint, once at least ``min_epoch_num`` epochs ran,
  training stops; otherwise it runs ``max_epoch_num`` epochs.

Data: the training and validation sets (``.dspf`` or the 12-column text feature file) are read once and
kept on the device (1 040 B per site for 13 x 16, plus the label); each epoch draws its order with
``torch.randperm`` from a CPU generator seeded with ``--tseed``, and every step gathers its batch on
the device.  A set that does not fit in free device memory is refused; there is no streaming."""
from __future__ import annotations

import os
import sys
import time

import numpy as np
import torch

KEYS = ("kmer", "base_means", "base_stds", "base_signal_lens", "signals")


def str2bool(v):
    return str(v).lower() in ("yes", "true", "t", "1", "y")


def ckpt_name(model_type, seq_len, signal_len, epoch):
    """The reference's checkpoint file name (``train.py:161-164``); ``epoch`` counts from 1."""
    return "{}.b{}_s{}_epoch{}.ckpt".format(model_type, seq_len, signal_len, epoch)


def load_feature_set(path, seq_len, signal_len, nthreads=None):
    """A ``.dspf`` or text feature file -> dict of CPU tensors (the five forward inputs, float32) plus
    ``labels`` (int64), in file order."""
    from . import feature_bin
    if feature_bin.is_feature_bin(path):
        reader = feature_bin.FeatureBinReader(path, seq_len, signal_len, pinned=False, slots=2, nthreads=nthreads)
    else:
        from .feature_io import FeatureFileReader
        reader = FeatureFileReader(path, seq_len, signal_len, pinned=False, slots=2, nthreads=nthreads)
    parts = {k: [] for k in KEYS + ("labels",)}
    for b in reader:
        for k, t in zip(KEYS + ("labels",), b.arrays() + (b.labels,)):
            parts[k].append(t[:b.n].clone())
    if not parts["labels"]:
        raise ValueError("%s holds no sites" % path)
    out = {k: torch.cat(v) for k, v in parts.items()}
    out["labels"] = out["labels"].to(torch.int64)
    return out


def bytes_per_site(seq_len, signal_len):
    return 4 * (4 * seq_len + seq_len * signal_len) + 8


def to_device(data, dev, what):
    n = data["labels"].shape[0]
    need = n * bytes_per_site(data["signals"].shape[1], data["signals"].shape[2])
    free, _ = torch.cuda.mem_get_info(dev)
    if need > free // 2:
        raise MemoryError("the %s set needs %.1f GB on the device (%d sites) but only %.1f GB are free; it must fit in "
                          "half of that, the rest is for the activations of training -- datasets larger than device "
                          "memory are not supported" % (what, need / 1e9, n, free / 1e9))
    return {k: v.to(dev) for k, v in data.items()}


def epoch_orders(n, tseed, epochs):
    """The site order of each epoch: ``torch.randperm`` from one CPU generator seeded with ``tseed``."""
    g = torch.Generator().manual_seed(int(tseed))
    return [torch.randperm(n, generator=g) for _ in range(epochs)]


def make_optimizer(name, params, lr):
    if name == "Adam":
        return torch.optim.Adam(params, lr=lr)
    if name == "RMSprop":
        return torch.optim.RMSprop(params, lr=lr)
    if name == "SGD":
        return torch.optim.SGD(params, lr=lr, momentum=0.8)
    raise ValueError("--optim_type must be Adam, RMSprop or SGD (Ranger is not available here)")


def evaluate(model, data, criterion, batch_size):
    """(mean loss, accuracy) of ``model`` in eval() mode over a device-resident set."""
    model.eval()
    n = data["labels"].shape[0]
    losses, correct = [], 0
    with torch.no_grad():
        for s in range(0, n, batch_size):
            x = [data[k][s:s + batch_size] for k in KEYS]
            y = data["labels"][s:s + batch_size]
            logits, probs = model(*x)
            losses.append(criterion(logits, y).item())
            correct += int((torch.max(probs, 1)[1] == y).sum().item())
    model.train()
    return float(np.mean(losses)), correct / n


def build_model(args, dev):
    from .models import ModelBiLSTM
    model = ModelBiLSTM(args.seq_len, args.signal_len, args.layernum1, args.layernum2, args.class_num,
                        args.dropout_rate, args.hid_rnn, args.n_vocab, args.n_embed, str2bool(args.is_base),
                        str2bool(args.is_signallen), args.model_type, device=dev.index, trainable=True)
    if args.init_model is not None:
        para = torch.load(args.init_model, map_location=torch.device("cpu"))
        d = model.state_dict()
        d.update(para)
        model.load_state_dict(d)
    return model.cuda(dev)


def train(args, log=print):
    if not torch.cuda.is_available():
        raise RuntimeError("train needs a CUDA device; this implementation has no CPU path")
    t0 = time.time()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    torch.manual_seed(args.tseed)
    torch.cuda.manual_seed(args.tseed)
    tr = to_device(load_feature_set(args.train_file, args.seq_len, args.signal_len), dev, "training")
    va = to_device(load_feature_set(args.valid_file, args.seq_len, args.signal_len), dev, "validation")
    n = tr["labels"].shape[0]
    model_dir = args.model_dir
    os.makedirs(model_dir, exist_ok=True)
    model = build_model(args, dev)
    criterion = torch.nn.CrossEntropyLoss(weight=torch.tensor([1.0, args.pos_weight], device=dev))
    optimizer = make_optimizer(args.optim_type, model.parameters(), args.lr)
    scheduler = torch.optim.lr_scheduler.StepLR(optimizer, step_size=2, gamma=0.1)
    orders = epoch_orders(n, args.tseed, args.max_epoch_num)
    steps = (n + args.batch_size - 1) // args.batch_size
    best, best_epoch, saved = 0.0, 0, []
    log("[train] %d training / %d validation sites, %d steps per epoch" % (n, va["labels"].shape[0], steps))
    model.train()
    for epoch in range(args.max_epoch_num):
        best_this_epoch, no_best_model, tlosses = 0.0, True, []
        order = orders[epoch].to(dev)
        te = time.time()
        for i in range(steps):
            idx = order[i * args.batch_size:(i + 1) * args.batch_size]
            x = [tr[k].index_select(0, idx) for k in KEYS]
            y = tr["labels"].index_select(0, idx)
            logits, _ = model(*x)
            loss = criterion(logits, y)
            tlosses.append(loss.detach())
            optimizer.zero_grad()
            loss.backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), 0.5)
            optimizer.step()
            if (i + 1) % args.step_interval == 0 or i == steps - 1:
                vloss, vacc = evaluate(model, va, criterion, args.batch_size)
                if vacc > best_this_epoch:
                    best_this_epoch = vacc
                    if best_this_epoch > best - 0.0002:
                        path = os.path.join(model_dir, ckpt_name(args.model_type, args.seq_len, args.signal_len, epoch + 1))
                        torch.save(model.state_dict(), path)
                        if path not in saved:
                            saved.append(path)
                        if best_this_epoch > best:
                            best, best_epoch = best_this_epoch, epoch + 1
                        no_best_model = False
                log("epoch [%d/%d], step [%d/%d], train loss %.4f, valid loss %.4f, valid acc %.4f, best %.4f (epoch %d)"
                    % (epoch + 1, args.max_epoch_num, i + 1, steps, torch.stack(tlosses).mean().item(), vloss, vacc,
                       best, best_epoch))
                tlosses = []
        log("[train] epoch %d: %.1f s" % (epoch + 1, time.time() - te))
        scheduler.step()
        if no_best_model and epoch >= args.min_epoch_num - 1:
            log("[train] early stop: no better validation accuracy in epoch %d" % (epoch + 1))
            break
    log("[train] best validation accuracy %.4f at epoch %d; %.1f s" % (best, best_epoch, time.time() - t0))
    return {"best_accuracy": best, "best_epoch": best_epoch, "checkpoints": saved}


def main(args):
    res = train(args)
    sys.stdout.flush()
    return res
