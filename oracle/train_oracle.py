"""ORACLE (test infrastructure, not product code): the reference forward in ``train()`` mode on torch's CPU
operators, differentiable, in float64.

``torch_oracle.forward`` with autograd enabled and the dropout masks as arguments (``models.py:178-240``:
nn.LSTM inter-layer dropout after every layer of a stack but the last, dropout -> fc1 -> dropout -> ReLU ->
fc2 in the head, none on the branch fc layers).  Stacks run one layer at a time so that the given
inter-layer masks can be applied; ``torch._VF.lstm`` over all layers would draw its own.  Masks hold
keep / (1 - p) and are multiplied in, which is what nn.Dropout computes; ``None`` = no dropout there.
Mask slots follow ``ModelBiLSTM.dropout_mask_shapes``."""
from __future__ import annotations

import torch
import torch.nn.functional as F


def _layer(x, sd, prefix, l, h0, c0):
    flat = []
    for sfx in ("", "_reverse"):
        flat += [sd["%s.weight_ih_l%d%s" % (prefix, l, sfx)], sd["%s.weight_hh_l%d%s" % (prefix, l, sfx)],
                 sd["%s.bias_ih_l%d%s" % (prefix, l, sfx)], sd["%s.bias_hh_l%d%s" % (prefix, l, sfx)]]
    out, _, _ = torch._VF.lstm(x, (h0, c0), flat, True, 1, 0.0, False, True, True)
    return out


def _stack(x, sd, prefix, layers, h0, c0, masks):
    for l in range(layers):
        x = _layer(x, sd, prefix, l, h0[2 * l:2 * l + 2], c0[2 * l:2 * l + 2])
        if l + 1 < layers and masks[l] is not None:
            x = x * masks[l]
    return x


def forward(sd, cfg, kmer, base_means, base_stds, base_signal_lens, signals, states, masks):
    """sd: state_dict of float64 CPU tensors (leaf tensors with requires_grad for gradients); cfg:
    ``model_oracle.make_cfg``; states: {"seq"|"signal"|"comb": (h0, c0)}; masks: the slot list.
    -> logits (differentiable)."""
    T, H, mod = cfg["seq_len"], cfg["hidden_size"], cfg["module"]
    L1, L2 = cfg["num_layers1"], cfg["num_layers2"]
    masks = [None if m is None else m.to(torch.float64) for m in masks]
    m_seq, m_sig = masks[:L2 - 1], masks[L2 - 1:2 * (L2 - 1)]
    m_comb, m1, m2 = masks[2 * (L2 - 1):2 * (L2 - 1) + L1 - 1], masks[-2], masks[-1]
    st = {k: (h.to(torch.float64), c.to(torch.float64)) for k, (h, c) in states.items()}
    parts = []
    if mod != "signal_bilstm":
        cols = []
        if cfg["is_base"]:
            cols.append(F.embedding(kmer.long(), sd["embed.weight"]))
        cols += [base_means.reshape(-1, T, 1).double(), base_stds.reshape(-1, T, 1).double()]
        if cfg["is_signallen"]:
            cols.append(base_signal_lens.reshape(-1, T, 1).double())
        x = _stack(torch.cat(cols, 2), sd, "lstm_seq", L2, *st["seq"], m_seq)
        parts.append(F.relu(F.linear(x, sd["fc_seq.weight"], sd["fc_seq.bias"])))
    if mod != "seq_bilstm":
        x = _stack(signals.double(), sd, "lstm_signal", L2, *st["signal"], m_sig)
        parts.append(F.relu(F.linear(x, sd["fc_signal.weight"], sd["fc_signal.bias"])))
    x = parts[0] if len(parts) == 1 else torch.cat(parts, 2)
    x = _stack(x, sd, "lstm_comb", L1, *st["comb"], m_comb)
    x = torch.cat((x[:, -1, :H], x[:, 0, H:]), 1)
    if m1 is not None:
        x = x * m1
    x = F.linear(x, sd["fc1.weight"], sd["fc1.bias"])
    if m2 is not None:
        x = x * m2
    return F.linear(F.relu(x), sd["fc2.weight"], sd["fc2.bias"])
