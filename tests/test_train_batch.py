"""The model-batched training step (dsp_train_forward_batch / dsp_train_backward_batch, forward_train_batch): every
model's logits and gradients bit-identical to its own one-model step (GPU), and the refusals before launch."""
import ctypes as C

import numpy as np
import pytest
import torch

from deepsignal_plant_b200 import _native, synthetic
from deepsignal_plant_b200.models import ModelBiLSTM, _TrainStep, forward_train_batch
from oracle import model_oracle

KEYS = ("kmer", "base_means", "base_stds", "base_signal_lens", "signals")


def _dev():
    return torch.device("cuda:0")


def _model(module, T, S, H, p, seed):
    torch.manual_seed(seed)
    return ModelBiLSTM(T, S, 3, 1, 2, p, H, 16, 4, True, True, module=module, precision="fp32",
                       trainable=True).cuda(0).train()


def _inputs(n, T, S, seed):
    f = synthetic.make_features(n, T, S, seed=seed)
    return [torch.from_numpy(f[k]).to(_dev()) for k in KEYS]


def _states(model, n, seed):
    cfg = model_oracle.make_cfg(model.seq_len, model.signal_len, 3, 1, 2, model.hidden_size, module=model.module)
    st = synthetic.make_states(cfg, n, seed=seed)
    keep = []
    ptrs = (C.c_void_p * 6)()
    for g, name in enumerate(("seq", "signal", "comb")):
        if name in st:
            h, c = (torch.from_numpy(x).to(_dev()).contiguous() for x in st[name])
            keep += [h, c]
            ptrs[2 * g], ptrs[2 * g + 1] = h.data_ptr(), c.data_ptr()
    return ptrs, keep


def _prep(model, x):
    return model._train_inputs(*x)


def _one_model(model, x, states, masks, seed, dlogits):
    params = model._train_params()
    handle = model._create_handle(_dev())
    logits = _TrainStep.apply(handle, _prep(model, x), states[0], states[1], masks, seed, *params)
    grads = torch.autograd.grad(logits, params, dlogits)
    return logits.detach(), grads


BATCH = [("both_bilstm", 13, 16, 256, 40), ("seq_bilstm", 13, 16, 256, 40), ("signal_bilstm", 13, 16, 256, 40),
         ("both_bilstm", 17, 20, 256, 24), ("both_bilstm", 13, 16, 32, 37), ("both_bilstm", 13, 16, 32, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("G", [1, 2, 3, 6, 8])
@pytest.mark.parametrize("p", [0.0, 0.5])
@pytest.mark.parametrize("module,T,S,H,n", BATCH)
def test_batched_step_equals_separate_steps_bit_for_bit(module, T, S, H, n, p, G):
    models = [_model(module, T, S, H, p, seed=100 + i) for i in range(G)]
    xs = [_inputs(n, T, S, seed=10 * n + i) for i in range(G)]
    states = [_states(m, n, seed=500 + i) for i, m in enumerate(models)]
    masks = [m.draw_dropout_masks(n, _dev()) for m in models]
    seeds = [1000 + i for i in range(G)]
    dls = [torch.randn(n, 2, generator=torch.Generator().manual_seed(7 + i)).to(_dev()) for i in range(G)]
    want = [_one_model(m, x, s, mk, sd, dl) for m, x, s, mk, sd, dl in zip(models, xs, states, masks, seeds, dls)]
    params = [p_ for m in models for p_ in m._train_params()]
    st = [p_ for s in states for p_ in s[0]]
    keep = [t for s in states for t in s[1]]
    logits = _TrainBatchStep_apply(models, [_prep(m, x) for m, x in zip(models, xs)], st, keep, masks, seeds, n, params)
    grads = torch.autograd.grad(logits, params, dls)
    npm = len(params) // G
    for i in range(G):
        assert torch.equal(logits[i].detach(), want[i][0]), "logits of model %d" % i
        for j, (a, b) in enumerate(zip(grads[i * npm:(i + 1) * npm], want[i][1])):
            assert torch.equal(a, b), "gradient %d of model %d" % (j, i)


def _TrainBatchStep_apply(models, inputs, states, keep, masks, seeds, n, params):
    from deepsignal_plant_b200.models import _TrainBatchStep
    handle = models[0]._create_handle(_dev())
    return _TrainBatchStep.apply(handle, len(models), n, inputs, states, keep, masks, seeds, *params)


@pytest.mark.gpu
def test_ten_adam_steps_batched_and_separate_leave_identical_parameters():
    G, n = 6, 96
    runs = []
    for batched in (True, False):
        models = [_model("both_bilstm", 13, 16, 64, 0.5, seed=200 + i) for i in range(G)]
        for i, m in enumerate(models):
            m.seed = 31 + i
            m.dropout_generator = torch.Generator(device=_dev()).manual_seed(77 + i)
        opts = [torch.optim.Adam(m.parameters(), lr=1e-3) for m in models]
        crit = torch.nn.CrossEntropyLoss(weight=torch.tensor([1.0, 2.0], device=_dev()))
        for step in range(10):
            xs = [_inputs(n, 13, 16, seed=1000 * step + i) for i in range(G)]
            ys = [torch.from_numpy(np.random.default_rng(step * 10 + i).integers(0, 2, n)).to(_dev()) for i in range(G)]
            for o in opts:
                o.zero_grad()
            if batched:
                logits = forward_train_batch(models, xs)
                sum(crit(lg, y) for lg, y in zip(logits, ys)).backward()
            else:
                for m, x, y in zip(models, xs, ys):
                    crit(m(*x)[0], y).backward()
            for m, o in zip(models, opts):
                torch.nn.utils.clip_grad_norm_(m.parameters(), 0.5)
                o.step()
        runs.append([[p.detach().clone() for p in m.parameters()] for m in models])
    for a, b in zip(*runs):
        for x, y in zip(a, b):
            assert torch.equal(x, y)


@pytest.mark.gpu
def test_forward_train_batch_cuts_groups_and_mixed_sizes():
    models = [_model("signal_bilstm", 13, 16, 32, 0.0, seed=300 + i) for i in range(11)]
    xs = [_inputs(20 if i % 3 else 21, 13, 16, seed=i) for i in range(11)]
    logits = forward_train_batch(models, xs)
    assert [lg.shape[0] for lg in logits] == [x[0].shape[0] for x in xs]
    for m, x, lg in zip(models, xs, logits):
        ref = _model("signal_bilstm", 13, 16, 32, 0.0, seed=0)
        ref.load_state_dict(m.state_dict())
        ref.seed, ref._calls = m.seed, m._calls - 1
        assert torch.equal(ref(*x)[0], lg)


@pytest.mark.gpu
def test_batched_step_has_the_launch_count_of_a_one_model_step():
    models = [_model("both_bilstm", 13, 16, 256, 0.5, seed=400 + i) for i in range(6)]
    xs = [_inputs(512, 13, 16, seed=i) for i in range(6)]
    handle_owner = models[0]
    handle_owner._create_handle(_dev())
    c0 = handle_owner.launch_count()
    handle_owner(*xs[0])[0].sum().backward()
    one = handle_owner.launch_count() - c0
    c1 = handle_owner.launch_count()
    sum(lg.sum() for lg in forward_train_batch(models, xs)).backward()
    batched = handle_owner.launch_count() - c1
    print("launches per training step: one model %d, six models batched %d" % (one, batched))
    assert one == batched and one > 0


@pytest.mark.gpu
def test_refusals_before_launch():
    models = [_model("signal_bilstm", 13, 16, 32, 0.0, seed=i) for i in range(9)]
    m0 = models[0]
    handle = m0._create_handle(_dev())
    L = _native.lib()
    n = 8
    params = [p for m in models for p in m._train_params()]
    npm = len(params) // 9
    nm = len(m0.dropout_mask_shapes(n))
    x = _prep(m0, _inputs(n, 13, 16, seed=0))
    inputs = (C.c_void_p * 45)(*[None if t is None else t.data_ptr() for _ in range(9) for t in x])
    arenas = [torch.empty(int(L.dsp_train_arena_bytes(handle, n)), dtype=torch.uint8, device=_dev()) for _ in range(9)]
    logits = [torch.empty(n, 2, device=_dev()) for _ in range(9)]
    pa = lambda ts: (C.c_void_p * max(1, len(ts)))(*[t.data_ptr() for t in ts])
    before = m0.launch_count()
    rc = L.dsp_train_forward_batch(handle, 9, pa(params), npm, inputs, None, (C.c_uint64 * 9)(*range(9)),
                                   (C.c_void_p * (9 * nm))(), n, pa(arenas), pa(logits), None)
    assert rc != 0 and b"models" in L.dsp_last_error()
    rc = L.dsp_train_forward_batch(handle, 2, pa(params), npm, inputs, None, (C.c_uint64 * 2)(1, 2),
                                   (C.c_void_p * (2 * nm))(), n, (C.c_void_p * 2)(arenas[0].data_ptr(), None), pa(logits), None)
    assert rc != 0 and b"arena of model 1" in L.dsp_last_error()
    rc = L.dsp_train_forward_batch(handle, 2, None, npm, inputs, None, (C.c_uint64 * 2)(1, 2),
                                   (C.c_void_p * (2 * nm))(), n, pa(arenas), pa(logits), None)
    assert rc != 0
    assert m0.launch_count() == before
    other = _model("signal_bilstm", 13, 16, 64, 0.0, seed=1)
    with pytest.raises(ValueError, match="equal configurations"):
        forward_train_batch([m0, other], [_inputs(n, 13, 16, seed=0)] * 2)
    cpu_model = ModelBiLSTM(13, 16, 3, 1, 2, 0.0, 32, module="signal_bilstm", trainable=True).train()
    with pytest.raises(RuntimeError, match="one CUDA device"):
        forward_train_batch([m0, cpu_model], [_inputs(n, 13, 16, seed=0)] * 2)
    assert m0.launch_count() == before
