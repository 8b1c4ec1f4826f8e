"""``denoise``: remove labelled positive samples that the data does not support, before ``train``.

Restates deepsignal-plant v0.1.6 ``denoise.py`` (``train_1time``, ``train_rounds``, ``clean_samples``, ``denoise``); the
reference's source is not part of this tree, so this module pins the contract below itself (DESIGN §9).

One iteration k works on the current sample set S (at the start: every sample of ``--train_file``, in file order).
For each round r of ``--rounds``, a permutation of S (drawn from ``(tseed, k, r)``) is cut into half A (its first
``|S| // 2`` samples) and half B (the rest); model (r, A) trains on A and scores B, model (r, B) trains on B and scores
A.  A model is a fresh ``ModelBiLSTM(..., trainable=True)`` trained for ``--epoch_num`` epochs with
CrossEntropyLoss(weight=[1, pos_weight]), Adam at ``--lr``, StepLR(step_size=2, gamma=0.1) per epoch and
``clip_grad_norm_(0.5)``; every epoch draws a fresh order of its half.  Nothing is validated during training.  Then it
scores its held-out half under ``eval()`` (the inference path ``train`` validates with): ``softmax[:, 1]``.  Every
sample gets ``rounds`` float32 scores per iteration; their mean and population std are taken in float64, adding the
scores in round order.

Cleaning: a label-1 sample is kept iff ``mean >= score_cf``; a label-0 sample is always kept with
``--is_filter_fn no`` and kept iff ``1 - mean >= score_cf`` with ``yes``.  The kept samples, in input order, are
written next to the input as ``<stem>.denoise_fp<k><ext>`` (``.denoise_fnp<k>`` with ``--is_filter_fn yes``; k counts
from 1), the previous iteration's file is deleted, and they become S.  Denoising stops after ``--iterations``
iterations or once ``left_ratio`` (kept / all positives) and ``left_ratio2`` (kept / all negatives, 1 with
``--is_filter_fn no``) both reach ``--kept_ratio``.  A text input gives its kept lines byte for byte; a ``.dspf`` input
gives a ``.dspf`` file whose rows are the input's kept rows bit for bit.

GPU work: the set is loaded to the device once and halves and batches are index tensors into it.  The ``2 * rounds``
models of one iteration train together: every step runs all of them through ``forward_train_batch`` (the
model-batched training kernels), so one set of launches carries up to DSP_TRAIN_MAX_MODELS models' batches of 512.

Determinism: every model's randomness (parameter initialisation, epoch orders from a CPU generator, dropout masks from
a CUDA generator, Philox seed of its initial states) comes from ``model_seed(tseed, k, r, half)``; the round
permutations from ``model_seed(tseed, k, r, 2)``.  The result depends on ``--tseed`` only, not on how the models are
grouped into batched steps (``max_models``).
"""
from __future__ import annotations

import hashlib
import os
import sys
import time

import numpy as np
import torch

from .train import KEYS, str2bool

HALF_A, HALF_B, PERMUTATION = 0, 1, 2


def model_seed(tseed, k, r, half):
    """The one seed formula of ``denoise``: 40 bits of SHA-256 over ``tseed:k:r:half`` (half 0 = A, 1 = B, 2 = the
    round's permutation)."""
    h = hashlib.sha256(("%d:%d:%d:%d" % (int(tseed), int(k), int(r), int(half))).encode()).digest()
    return int.from_bytes(h[:5], "little")


def round_halves(n, tseed, k, r):
    """(A, B): positions into S of round r of iteration k; A = the first ``n // 2`` of a permutation, B the rest."""
    g = torch.Generator().manual_seed(model_seed(tseed, k, r, PERMUTATION))
    perm = torch.randperm(n, generator=g)
    return perm[:n // 2], perm[n // 2:]


def score_stats(scores):
    """(rounds, n) float32 scores -> (mean, population std) in float64, summed in round order."""
    s = np.asarray(scores, dtype=np.float32).astype(np.float64)
    acc = np.zeros(s.shape[1], np.float64)
    for row in s:
        acc += row
    mean = acc / s.shape[0]
    var = np.zeros(s.shape[1], np.float64)
    for row in s:
        var += (row - mean) ** 2
    return mean, np.sqrt(var / s.shape[0])


def clean(labels, mean, score_cf, is_filter_fn):
    """-> (keep mask, counts): the cleaning rule on one iteration's mean scores."""
    labels = np.asarray(labels)
    mean = np.asarray(mean, dtype=np.float64)
    pos, neg = labels == 1, labels != 1
    keep = np.ones(labels.shape[0], bool)
    keep[pos] = mean[pos] >= score_cf
    if is_filter_fn:
        keep[neg] = 1.0 - mean[neg] >= score_cf
    n_pos, n_neg = int(pos.sum()), int(neg.sum())
    kept_pos, kept_neg = int((keep & pos).sum()), int((keep & neg).sum())
    left_ratio = kept_pos / n_pos if n_pos else 0.0
    left_ratio2 = (kept_neg / n_neg if n_neg else 1.0) if is_filter_fn else 1.0
    return keep, dict(positives=n_pos, negatives=n_neg, kept_positives=kept_pos, kept_negatives=kept_neg,
                      left_ratio=left_ratio, left_ratio2=left_ratio2)


def should_stop(counts, kept_ratio):
    return counts["left_ratio"] >= kept_ratio and counts["left_ratio2"] >= kept_ratio


def output_path(train_file, k, is_filter_fn):
    """``<stem>.denoise_fp<k><ext>`` (``denoise_fnp`` with is_filter_fn), k counting from 1."""
    stem, ext = os.path.splitext(train_file)
    return "%s.denoise_%s%d%s" % (stem, "fnp" if is_filter_fn else "fp", k, ext)


def check_input(train_file):
    if train_file.endswith(".gz"):
        raise ValueError("denoise reads plain text or .dspf feature files; decompress %s first" % train_file)
    if not os.path.exists(train_file):
        raise FileNotFoundError(train_file)


def write_kept(src, dst, rows):
    """The input's rows at the sorted original indices ``rows`` -> ``dst``: text lines byte for byte, or a .dspf file
    whose arrays, labels and sample-info columns are the input's rows bit for bit."""
    from . import feature_bin
    if feature_bin.is_feature_bin(src):
        reader = feature_bin.FeatureBinReader(src, pinned=False, slots=2)
        keep = np.zeros(reader.total_sites, bool)
        keep[rows] = True
        g = 0
        with feature_bin.FeatureBinWriter(dst, reader.T, reader.S) as w:
            for b in reader:
                sel = np.nonzero(keep[g:g + b.n])[0]
                g += b.n
                if sel.size == 0:
                    continue
                off = b.info_off[:b.n + 1]
                parts = [bytes(b.info_text[off[i]:off[i + 1]]) for i in sel]
                new_off = np.zeros(sel.size + 1, np.int64)
                new_off[1:] = np.cumsum([len(p) for p in parts])
                w.write(*(t.numpy()[sel] for t in (b.kmer, b.base_means, b.base_stds, b.base_signal_lens, b.signals,
                                                   b.labels)), b"".join(parts), new_off)
        return
    rows = np.asarray(rows, np.int64)
    j = 0
    with open(src, "rb") as fi, open(dst, "wb") as fo:
        i = 0
        for line in fi:
            if not line.strip():
                continue
            if j < rows.size and rows[j] == i:
                fo.write(line)
                j += 1
            i += 1
    if j != rows.size:
        raise ValueError("%s holds fewer sites than were loaded from it" % src)


def build_model(args, dev, seed):
    from .models import ModelBiLSTM
    with torch.random.fork_rng(devices=[]):        # parameter initialisation draws from the CPU generator only
        torch.default_generator.manual_seed(seed)
        model = ModelBiLSTM(args.seq_len, args.signal_len, args.layernum1, args.layernum2, args.class_num,
                            args.dropout_rate, args.hid_rnn, args.n_vocab, args.n_embed, str2bool(args.is_base),
                            str2bool(args.is_signallen), args.model_type, device=dev.index, seed=seed, trainable=True)
    model = model.cuda(dev)
    model.dropout_generator = torch.Generator(device=dev).manual_seed(seed)
    return model


def train_and_score(data, S, k, args, dev, log, max_models):
    """One iteration's ``2 * rounds`` models, trained together -> (rounds, |S|) float32 scores of the held-out
    halves."""
    from .models import forward_train_batch
    R, bs = args.rounds, args.batch_size
    n = S.shape[0]
    jobs = []      # (round, half, model, train positions, held-out positions, CPU generator)
    for r in range(R):
        A, B = round_halves(n, args.tseed, k, r)
        for half, (tr, ho) in ((HALF_A, (A, B)), (HALF_B, (B, A))):
            seed = model_seed(args.tseed, k, r, half)
            jobs.append((r, half, build_model(args, dev, seed), tr, ho, torch.Generator().manual_seed(seed)))
    weight = torch.tensor([1.0, args.pos_weight], device=dev)
    criterion = torch.nn.CrossEntropyLoss(weight=weight)
    opts = [torch.optim.Adam(j[2].parameters(), lr=args.lr) for j in jobs]
    scheds = [torch.optim.lr_scheduler.StepLR(o, step_size=2, gamma=0.1) for o in opts]
    models = [j[2] for j in jobs]
    for m in models:
        m.train()
    group = max(1, int(max_models))
    for epoch in range(args.epoch_num):
        orders = [S[j[3][torch.randperm(j[3].shape[0], generator=j[5])].to(dev)] for j in jobs]
        steps = [(o.shape[0] + bs - 1) // bs for o in orders]
        losses = [[] for _ in jobs]
        for i in range(max(steps)):
            active = [q for q in range(len(jobs)) if i < steps[q]]
            idx = [orders[q][i * bs:(i + 1) * bs] for q in active]
            for c in range(0, len(active), group):
                part = active[c:c + group]
                sel = idx[c:c + group]
                logits = forward_train_batch([models[q] for q in part],
                                             [[data[key].index_select(0, ix) for key in KEYS] for ix in sel])
                loss = [criterion(lg, data["labels"].index_select(0, ix)) for lg, ix in zip(logits, sel)]
                for q in part:
                    opts[q].zero_grad()
                sum(loss).backward()
                for q, lo in zip(part, loss):
                    torch.nn.utils.clip_grad_norm_(models[q].parameters(), 0.5)
                    opts[q].step()
                    losses[q].append(lo.detach())
            if (i + 1) % args.step_interval == 0 or i == max(steps) - 1:
                msg = ", ".join("r%d%s %.4f" % (j[0], "AB"[j[1]], torch.stack(lq).mean().item())
                                for j, lq in zip(jobs, losses) if lq)
                log("[denoise] iteration %d, epoch [%d/%d], step [%d/%d], train loss: %s"
                    % (k + 1, epoch + 1, args.epoch_num, i + 1, max(steps), msg))
                losses = [[] for _ in jobs]
        for s in scheds:
            s.step()
    scores = np.zeros((R, n), np.float32)
    with torch.no_grad():
        for (r, _, model, _, ho, _) in jobs:
            model.eval()
            rows = S[ho.to(dev)]
            out = []
            for s in range(0, rows.shape[0], bs):
                ix = rows[s:s + bs]
                out.append(model(*[data[key].index_select(0, ix) for key in KEYS])[1][:, 1])
            scores[r, ho.numpy()] = torch.cat(out).cpu().numpy()
    return scores


def denoise(args, log=print, max_models=None):
    """Run ``denoise``; -> dict(path = the final cleaned file, iterations = per-iteration counts, scores = per-iteration
    (rounds, |S|) float32 score arrays, samples = per-iteration original indices of S).  ``max_models`` (tests only)
    caps the models per batched training step."""
    from . import _native
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        raise RuntimeError("multi-GPU denoise is not supported; run it as one process (without torchrun)")
    if args.rounds < 1 or args.iterations < 1:
        raise ValueError("--rounds and --iterations must be at least 1")
    check_input(args.train_file)
    from .train import load_feature_set, to_device
    host = load_feature_set(args.train_file, args.seq_len, args.signal_len)
    labels = host["labels"].numpy()
    if labels.shape[0] < 2:
        raise ValueError("%s holds %d site(s); denoise needs at least 2" % (args.train_file, labels.shape[0]))
    if not (labels == 1).any():
        raise ValueError("%s holds no label-1 site; there is nothing to denoise" % args.train_file)
    if not torch.cuda.is_available():
        raise RuntimeError("denoise needs a CUDA device; this implementation has no CPU path")
    is_filter_fn = str2bool(args.is_filter_fn)
    max_models = _native.TRAIN_MAX_MODELS if max_models is None else int(max_models)
    t0 = time.time()
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    data = to_device(host, dev, "training")
    S = np.arange(labels.shape[0], dtype=np.int64)
    res = dict(path=None, iterations=[], scores=[], samples=[])
    for k in range(args.iterations):
        if S.size < 2 or not (labels[S] == 1).any():
            log("[denoise] %d sites (%d positive) left: stopping" % (S.size, int((labels[S] == 1).sum())))
            break
        ti = time.time()
        scores = train_and_score(data, torch.from_numpy(S).to(dev), k, args, dev, log, max_models)
        mean, std = score_stats(scores)
        keep, counts = clean(labels[S], mean, args.score_cf, is_filter_fn)
        S_next = S[keep]
        path = output_path(args.train_file, k + 1, is_filter_fn)
        write_kept(args.train_file, path, S_next)
        if res["path"] is not None and res["path"] != args.train_file:
            os.remove(res["path"])
        counts.update(iteration=k + 1, path=path, seconds=time.time() - ti)
        res["path"] = path
        res["iterations"].append(counts)
        res["scores"].append(scores)
        res["samples"].append(S)
        log("[denoise] iteration %d: %d positive, %d negative sites; kept %d positive (left_ratio %.4f), %d negative "
            "(left_ratio2 %.4f) -> %s; %.1f s" % (k + 1, counts["positives"], counts["negatives"],
                                                  counts["kept_positives"], counts["left_ratio"],
                                                  counts["kept_negatives"], counts["left_ratio2"], path,
                                                  counts["seconds"]))
        S = S_next
        if should_stop(counts, args.kept_ratio):
            log("[denoise] left_ratio and left_ratio2 reached kept_ratio %.4f: stopping" % args.kept_ratio)
            break
    log("[denoise] %s; %.1f s" % (res["path"], time.time() - t0))
    return res


def main(args):
    res = denoise(args)
    sys.stdout.flush()
    return res
