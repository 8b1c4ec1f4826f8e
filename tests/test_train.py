"""Training: the ``train`` command's host logic (CPU) and the fp32 training kernels against the float64 autograd
oracle (``oracle/train_oracle.py``, GPU)."""
import os

import numpy as np
import pytest
import torch

from deepsignal_plant_b200 import cli, synthetic
from deepsignal_plant_b200 import train as tr
from deepsignal_plant_b200.models import ModelBiLSTM
from oracle import model_oracle, train_oracle

KEYS = tr.KEYS


# ---- fixtures --------------------------------------------------------------------------------------------------
def labelled_features(n, T=13, S=16, seed=0, shift=5.0):
    """Synthetic sites; label-1 sites have their centre base's mean and signal shifted up (by 5 standard deviations of
    the means, so that the classes are separable)."""
    f = synthetic.make_features(n, T, S, seed=seed)
    labels = np.random.default_rng(seed + 1).integers(0, 2, n).astype(np.int32)
    f["base_means"][labels == 1, T // 2] += shift
    f["signals"][labels == 1, T // 2, :] += shift
    return f, labels


def write_pair(tmp_path, n, seed, T=13, S=16, name="set"):
    """The same labelled sites as a text feature file and as a .dspf file."""
    from deepsignal_plant_b200.feature_bin import pack_feature_file
    from deepsignal_plant_b200.feature_io import features_to_str
    f, labels = labelled_features(n, T, S, seed)
    f["base_means"] = np.round(f["base_means"].astype(np.float64), 6).astype(np.float32)
    txt = tmp_path / (name + ".tsv")
    with open(txt, "w") as fh:
        for i in range(n):
            info = "chr1\t%d\t+\t%d\tread%d\tt" % (1000 + i, 1000 + i, i)
            fh.write(features_to_str(info, f["kmer"][i], f["base_means"][i], f["base_stds"][i], f["base_signal_lens"][i],
                                     f["signals"][i], labels[i]) + "\n")
    binp = tmp_path / (name + ".dspf")
    pack_feature_file(str(txt), str(binp))
    return str(txt), str(binp), labels


def train_args(*extra):
    return cli.build_parser().parse_args(["train", "--train_file", "t", "--valid_file", "v", "--model_dir", "m"] + list(extra))


# ---- CPU -------------------------------------------------------------------------------------------------------
def test_train_flags_parse_with_reference_defaults():
    a = train_args()
    want = dict(model_type="both_bilstm", seq_len=13, signal_len=16, layernum1=3, layernum2=1, class_num=2,
                dropout_rate=0.5, n_vocab=16, n_embed=4, is_base="yes", is_signallen="yes", hid_rnn=256,
                optim_type="Adam", batch_size=512, lr=0.001, max_epoch_num=10, min_epoch_num=5, step_interval=100,
                pos_weight=1.0, init_model=None, tseed=1234)
    for k, v in want.items():
        assert getattr(a, k) == v, k
    assert (a.train_file, a.valid_file, a.model_dir) == ("t", "v", "m")


def test_dspf_and_text_training_inputs_are_identical(tmp_path):
    txt, binp, labels = write_pair(tmp_path, 300, seed=7)
    a = tr.load_feature_set(txt, 13, 16)
    b = tr.load_feature_set(binp, 13, 16)
    for k in KEYS + ("labels",):
        assert a[k].dtype == b[k].dtype and torch.equal(a[k], b[k]), k
    assert np.array_equal(a["labels"].numpy(), labels)


def test_epoch_order_is_deterministic_under_tseed():
    a = tr.epoch_orders(1000, 1234, 3)
    b = tr.epoch_orders(1000, 1234, 3)
    c = tr.epoch_orders(1000, 99, 3)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert not torch.equal(a[0], a[1]) and not torch.equal(a[0], c[0])
    assert torch.equal(torch.sort(a[2]).values, torch.arange(1000))


def test_checkpoint_names_follow_the_reference():
    assert tr.ckpt_name("both_bilstm", 13, 16, 1) == "both_bilstm.b13_s16_epoch1.ckpt"
    assert tr.ckpt_name("seq_bilstm", 17, 20, 10) == "seq_bilstm.b17_s20_epoch10.ckpt"


def test_saved_checkpoint_loads_into_an_eval_module(tmp_path):
    torch.manual_seed(2)
    a = ModelBiLSTM(hidden_size=32, trainable=True)
    with torch.no_grad():
        for p in a.parameters():
            p.mul_(1.5)
    path = tmp_path / tr.ckpt_name("both_bilstm", 13, 16, 3)
    torch.save(a.state_dict(), path)
    b = ModelBiLSTM(hidden_size=32).eval()
    d = b.state_dict()
    d.update(torch.load(path, map_location=torch.device("cpu")))
    b.load_state_dict(d)
    assert all(torch.equal(v, b.state_dict()[k]) for k, v in a.state_dict().items())
    assert not b.training


def test_train_oracle_without_dropout_is_the_inference_oracle():
    from oracle import torch_oracle
    torch.manual_seed(4)
    m = ModelBiLSTM(hidden_size=32)
    cfg = model_oracle.make_cfg(hidden_size=32)
    f, _ = labelled_features(9, seed=2)
    st = {k: tuple(torch.from_numpy(x) for x in v) for k, v in synthetic.make_states(cfg, 9).items()}
    x = [torch.from_numpy(f[k]) for k in KEYS]
    want = torch_oracle.forward(m.state_dict(), cfg, *x, st)[0]
    got = train_oracle.forward({k: v.double() for k, v in m.state_dict().items()}, cfg, *x, st, [None] * 4)
    assert float((got - want.double()).abs().max()) < 1e-5


def test_dropout_mask_slots():
    m = ModelBiLSTM(hidden_size=32, num_layers1=3, num_layers2=2, dropout_rate=0.5)
    assert m.dropout_mask_shapes(5) == [(5, 13, 32), (5, 13, 32), (5, 13, 64), (5, 13, 64), (5, 64), (5, 32)]
    m = ModelBiLSTM(hidden_size=32, module="signal_bilstm")
    assert m.dropout_mask_shapes(5) == [(5, 13, 64), (5, 13, 64), (5, 64), (5, 32)]


# ---- GPU: gradient parity against the float64 oracle ----------------------------------------------------------
def _dev():
    return torch.device("cuda:0")


def _model(module, T, S, H, p, seed=1234, L1=3):
    torch.manual_seed(seed)
    return ModelBiLSTM(T, S, L1, 1, 2, p, H, 16, 4, True, True, module=module, precision="fp32",
                       state_mode="init_hidden", trainable=True).cuda(0)


def _serve_states(model, states):
    order = iter(["seq", "signal", "comb"] if model.module == "both_bilstm" else
                 (["seq", "comb"] if model.module == "seq_bilstm" else ["signal", "comb"]))
    model.init_hidden = lambda b, l, h: tuple(torch.from_numpy(x).to(_dev()) for x in states[next(order)])


def _inputs(f):
    return [torch.from_numpy(f[k]).to(_dev()) for k in KEYS]


def _oracle(model, f, states, masks, dlogits):
    cfg = model_oracle.make_cfg(model.seq_len, model.signal_len, model.num_layers1, model.num_layers2, 2,
                                model.hidden_size, module=model.module)
    sd = {k: v.detach().cpu().double().requires_grad_() for k, v in model.state_dict().items()}
    st = {k: (torch.from_numpy(h), torch.from_numpy(c)) for k, (h, c) in states.items()}
    logits = train_oracle.forward(sd, cfg, *(torch.from_numpy(f[k]) for k in KEYS), st,
                                  [None if m is None else m.cpu() for m in masks])
    logits.backward(dlogits.cpu().double())
    return logits.detach(), {k: v.grad for k, v in sd.items()}


PARITY = [("both_bilstm", 13, 16, 256, 40), ("seq_bilstm", 13, 16, 256, 40), ("signal_bilstm", 13, 16, 256, 40),
          ("both_bilstm", 17, 20, 256, 24), ("both_bilstm", 13, 16, 32, 37), ("both_bilstm", 13, 16, 32, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.0, 0.5])
@pytest.mark.parametrize("module,T,S,H,n", PARITY)
def test_gradients_match_float64_oracle(module, T, S, H, n, p):
    model = _model(module, T, S, H, p).train()
    f, labels = labelled_features(n, T, S, seed=n)
    cfg = model_oracle.make_cfg(T, S, 3, 1, 2, H, module=module)
    states = synthetic.make_states(cfg, n, seed=77)
    _serve_states(model, states)
    logits, probs = model(*_inputs(f))
    dlogits = torch.randn(n, 2, generator=torch.Generator().manual_seed(5)).to(_dev())
    logits.backward(dlogits)
    want_logits, want_grads = _oracle(model, f, states, model.last_dropout_masks, dlogits)
    lerr = float((logits.detach().cpu().double() - want_logits).abs().max())
    assert torch.allclose(probs, torch.softmax(logits, 1))
    worst, worst_name = 0.0, ""
    for name, prm in model.named_parameters():
        g, w = prm.grad.cpu().double(), want_grads[name]
        scale = float(w.abs().max()) or 1.0
        rel = float((g - w).abs().max()) / scale
        if rel > worst:
            worst, worst_name = rel, name
    print("train parity %s T=%d S=%d H=%d n=%d p=%.1f: max|dlogits| %.2e, worst grad err %.2e x max|g| (%s)"
          % (module, T, S, H, n, p, lerr, worst, worst_name))
    assert lerr < 1e-5
    assert worst < 1e-4, worst_name


@pytest.mark.gpu
def test_repeated_backward_is_bit_identical():
    model = _model("both_bilstm", 13, 16, 256, 0.5).train()
    f, _ = labelled_features(600, seed=3)
    logits, _ = model(*_inputs(f))
    loss = torch.nn.functional.cross_entropy(logits, torch.ones(600, dtype=torch.long, device=_dev()))
    loss.backward(retain_graph=True)
    first = [p.grad.clone() for p in model.parameters()]
    model.zero_grad()
    loss.backward()
    for a, p in zip(first, model.parameters()):
        assert torch.equal(a, p.grad)


@pytest.mark.gpu
def test_two_forwards_one_backward_is_the_sum_of_single_backwards():
    model = _model("both_bilstm", 13, 16, 64, 0.0).train()
    fa, _ = labelled_features(50, seed=4)
    fb, _ = labelled_features(70, seed=5)
    cfg = model_oracle.make_cfg(hidden_size=64)
    sa, sb = synthetic.make_states(cfg, 50, seed=1), synthetic.make_states(cfg, 70, seed=2)
    single = []
    for f, s in ((fa, sa), (fb, sb)):
        model.zero_grad()
        _serve_states(model, s)
        model(*_inputs(f))[0].square().sum().backward()
        single.append([p.grad.clone() for p in model.parameters()])
    model.zero_grad()
    _serve_states(model, sa)
    la = model(*_inputs(fa))[0]
    _serve_states(model, sb)
    lb = model(*_inputs(fb))[0]
    (la.square().sum() + lb.square().sum()).backward()
    for a, b, p in zip(single[0], single[1], model.parameters()):
        assert torch.allclose(p.grad, a + b, rtol=1e-5, atol=1e-6 * float((a + b).abs().max()))


@pytest.mark.gpu
def test_adam_steps_track_the_oracle_loss_trajectory():
    n, H = 128, 64
    model = _model("both_bilstm", 13, 16, H, 0.0).train()
    f, labels = labelled_features(n, seed=9)
    cfg = model_oracle.make_cfg(hidden_size=H)
    states = synthetic.make_states(cfg, n, seed=8)
    y = torch.from_numpy(labels.astype(np.int64))
    sd = {k: v.detach().cpu().double().requires_grad_() for k, v in model.state_dict().items()}
    names = [k for k, _ in model.named_parameters()]
    opt_o = torch.optim.Adam([sd[k] for k in names], lr=1e-3)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    st = {k: (torch.from_numpy(h), torch.from_numpy(c)) for k, (h, c) in states.items()}
    x_cpu = [torch.from_numpy(f[k]) for k in KEYS]
    got, want = [], []
    for _ in range(20):
        _serve_states(model, states)
        opt.zero_grad()
        loss = torch.nn.functional.cross_entropy(model(*_inputs(f))[0], y.to(_dev()))
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 0.5)
        opt.step()
        got.append(loss.item())
        opt_o.zero_grad()
        lo = torch.nn.functional.cross_entropy(train_oracle.forward(sd, cfg, *x_cpu, st, [None] * 4), y)
        lo.backward()
        torch.nn.utils.clip_grad_norm_([sd[k] for k in names], 0.5)
        opt_o.step()
        want.append(lo.item())
    rel = max(abs(a - b) / abs(b) for a, b in zip(got, want))
    print("20 Adam steps: loss %.6f -> %.6f, oracle %.6f -> %.6f, worst relative gap %.2e" % (got[0], got[-1], want[0],
                                                                                             want[-1], rel))
    assert rel < 1e-4


@pytest.mark.gpu
def test_dropout_keep_fraction():
    model = _model("both_bilstm", 13, 16, 256, 0.5)
    masks = model.draw_dropout_masks(200, _dev())
    kept = sum(int((m > 0).sum()) for m in masks if m is not None)
    total = sum(m.numel() for m in masks if m is not None)
    assert total >= 10 ** 6
    assert abs(kept / total - 0.5) < 4 * (0.25 / total) ** 0.5
    assert all(float(m.max()) == 2.0 for m in masks if m is not None)


@pytest.mark.gpu
def test_eval_after_training_matches_oracle_in_fp32_and_fp16():
    model = _model("both_bilstm", 13, 16, 256, 0.5).train()
    f, labels = labelled_features(512, seed=11)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    y = torch.from_numpy(labels.astype(np.int64)).to(_dev())
    for _ in range(5):
        opt.zero_grad()
        torch.nn.functional.cross_entropy(model(*_inputs(f))[0], y).backward()
        opt.step()
    cfg = model_oracle.make_cfg()
    states = synthetic.make_states(cfg, 512, seed=6)
    params = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    want = model_oracle.forward(params, cfg, *(f[k] for k in KEYS), states)[1]
    for precision in ("fp32", "fp16"):
        ev = ModelBiLSTM(13, 16, 3, 1, 2, 0, 256, precision=precision).cuda(0)
        ev.load_state_dict(model.state_dict())
        ev.eval()
        _serve_states(ev, states)
        probs = ev(*_inputs(f))[1].cpu().numpy()
        err = float(np.abs(probs - want).max())
        print("eval after training [%s]: max|dprob| %.2e" % (precision, err))
        assert err < 1e-3
        assert (probs.argmax(1) == want.argmax(1)).mean() >= 1.0 - 1.5 / 512


@pytest.mark.gpu
def test_train_command_end_to_end_then_call_mods(tmp_path):
    _, tr_bin, _ = write_pair(tmp_path, 16384, seed=21, name="train")
    _, va_bin, va_labels = write_pair(tmp_path, 2048, seed=22, name="valid")
    mdir = tmp_path / "models"
    args = cli.build_parser().parse_args(["train", "--train_file", tr_bin, "--valid_file", va_bin, "--model_dir", str(mdir)])
    res = tr.train(args)
    print("train end to end:", res)
    assert res["best_accuracy"] >= 0.95
    names = sorted(os.listdir(mdir))
    assert names and all(n.startswith("both_bilstm.b13_s16_epoch") and n.endswith(".ckpt") for n in names)
    best = os.path.join(mdir, tr.ckpt_name("both_bilstm", 13, 16, res["best_epoch"]))
    out = tmp_path / "calls.tsv"
    assert cli.main(["call_mods", "-i", va_bin, "-m", best, "-o", str(out)]) == 0
    called = np.array([int(line.split("\t")[8]) for line in open(out)])
    acc = float((called == va_labels).mean())
    print("call_mods with the trained checkpoint: accuracy %.4f (training reported %.4f)" % (acc, res["best_accuracy"]))
    assert len(called) == 2048 and acc >= 0.95
