"""GPU: the CUDA path (through the C ABI) against the reference-generated fixtures and the
numpy oracle.  Tolerances are the ones BASELINE.json's north_star states: probabilities
within 1e-3 absolute, labels >= 99.99 % identical; the fp32 path is held to 2e-5."""
import os

import numpy as np
import pytest
import torch

import cases
from deepsignal_plant_b200 import call_modifications as cm
from deepsignal_plant_b200 import synthetic
from oracle import model_oracle

pytestmark = pytest.mark.gpu

PROB_TOL = 1e-3          # north_star: prob_0/prob_1 within 1e-3 absolute
LABEL_AGREEMENT = 0.9999  # north_star: called labels >= 99.99 % identical
FP32_TOL = 2e-5


def run_case(case, precision, max_batch=4096):
    dev = torch.device("cuda:0")
    model = cases.build_model(case["entry"], precision=precision, max_batch=max_batch).cuda(0)
    cases.inject_states(model, case["states"], dev)
    f = case["feats"]
    args = [torch.from_numpy(f[k]).to(dev) for k in cases.FEATURE_KEYS]
    logits, probs = model(*args)
    torch.cuda.synchronize()
    assert model.launch_count() > 0
    return logits.cpu().numpy(), probs.cpu().numpy(), model.last_labels.cpu().numpy(), model


def check(case, logits, probs, labels, prob_tol, min_agree):
    gold = case["probs"]
    assert probs.shape == gold.shape and np.isfinite(probs).all()
    err = np.abs(probs - gold).max()
    agree = (probs.argmax(1) == gold.argmax(1)).mean()
    assert err <= prob_tol, "max |dprob| %.3e" % err
    assert agree >= min_agree, "label agreement %.5f" % agree
    assert (labels == probs.argmax(1)).all()
    np.testing.assert_allclose(probs.sum(1), 1.0, atol=1e-5)
    return err, agree


@pytest.mark.parametrize("name", cases.FORWARD_CASES)
def test_fp32_path_matches_reference(name):
    case = cases.load_case(name)
    logits, probs, labels, _ = run_case(case, "fp32")
    err, agree = check(case, logits, probs, labels, FP32_TOL, 1.0 if case["entry"]["n"] < 1000 else LABEL_AGREEMENT)
    assert np.abs(logits - case["logits"]).max() < 1e-4
    print("%s fp32: max|dprob|=%.2e agreement=%.5f" % (name, err, agree))


FP16_CASES = [n for n in cases.FORWARD_CASES if cases.MANIFEST["forward"][n]["ctor"]["hidden_size"] == 256]


@pytest.mark.parametrize("name", FP16_CASES)
def test_fp16_tensor_core_path_matches_reference(name):
    case = cases.load_case(name)
    logits, probs, labels, _ = run_case(case, "fp16")
    err, agree = check(case, logits, probs, labels, PROB_TOL, LABEL_AGREEMENT)
    print("%s fp16: max|dprob|=%.2e agreement=%.5f" % (name, err, agree))


@pytest.mark.parametrize("dual", ["0", "1", "fused"])
def test_fp16_both_branch_kernels_match_reference(dual, monkeypatch):
    # hidden-128 layers: by default both branches + their fc layers run as ONE launch (branch_fused_kernel);
    # DSP_B200_BRANCH_DUAL (read at handle creation) keeps the separate launches: 0 = one CTA pair per direction
    # (layer_kernel), 1 = both directions as two chains (branch_kernel), each followed by the fc launches
    if dual == "fused":
        monkeypatch.delenv("DSP_B200_BRANCH_DUAL", raising=False)
    else:
        monkeypatch.setenv("DSP_B200_BRANCH_DUAL", dual)
    for name in ("both_13_16_s2", "both_17_20_s1234"):
        case = cases.slice_case(cases.load_case(name), 3000)
        logits, probs, labels, model = run_case(case, "fp16")
        check(case, logits, probs, labels, PROB_TOL, 1.0 - 1.5 / 3000)          # at most one flip in 3 000 sites
        assert model.launch_count() == {"0": 9, "1": 9, "fused": 6}[dual]      # prep, branches(+fc), 3 x lstm_comb, head


def test_fp16_full_batch_is_batching_and_order_invariant():
    # BASELINE.json configs[1] batch (65 536 sites): size-independent properties of a per-site classifier
    # with explicit states -- sites are independent (models.py:178-240 has no cross-site op), so splitting
    # the batch or permuting the sites must give bit-identical probabilities; a 2 048-site sample is also
    # checked against the oracle.
    n = 65536
    cfg = model_oracle.make_cfg()
    feats = synthetic.make_features(n, 13, 16, seed=123)
    states = synthetic.make_states(cfg, n, seed=321)
    entry = cases.MANIFEST["forward"]["both_13_16_s1234"]
    dev = torch.device("cuda:0")
    model = cases.build_model(entry, precision="fp16", max_batch=n).cuda(0)

    def run(idx):
        f = {k: v[idx] for k, v in feats.items()}
        st = {g: tuple(np.ascontiguousarray(x[:, idx]) for x in hc) for g, hc in states.items()}
        cases.inject_states(model, st, dev)
        _, probs = model(*(torch.from_numpy(np.ascontiguousarray(f[k])).to(dev) for k in cases.FEATURE_KEYS))
        return probs.cpu().numpy(), model.last_labels.cpu().numpy()
    full, labels = run(np.arange(n))
    assert np.isfinite(full).all() and (labels == full.argmax(1)).all()
    half_a, _ = run(np.arange(0, 30001))                   # ragged split, different tile alignment of every site after it
    half_b, _ = run(np.arange(30001, n))
    assert np.array_equal(np.concatenate([half_a, half_b]), full)
    perm = np.random.default_rng(5).permutation(n)
    shuffled, _ = run(perm)
    assert np.array_equal(shuffled, full[perm])
    sample = np.arange(0, n, 32)
    params = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    want = model_oracle.forward(params, cfg, *(feats[k][sample] for k in cases.FEATURE_KEYS),
                                {g: tuple(x[:, sample] for x in hc) for g, hc in states.items()})[1]
    assert np.abs(full[sample] - want).max() <= PROB_TOL
    assert int((full[sample].argmax(1) != want.argmax(1)).sum()) <= 1            # 2 048 sites: at most one flip


def test_repacking_after_load_state_dict_replaces_the_weights():
    # call_modifications.py:219-223 loads a checkpoint into an already constructed model: the second
    # pack must replace (and free) the first arena
    a = cases.slice_case(cases.load_case("both_13_16_s1"), 1500)
    b = cases.slice_case(cases.load_case("both_13_16_s2"), 1500)
    dev = torch.device("cuda:0")
    model = cases.build_model(a["entry"], precision="fp16").cuda(0)
    for case in (a, b, a):
        model.load_state_dict({k: torch.from_numpy(v) for k, v in case["params"].items()})
        cases.inject_states(model, case["states"], dev)
        _, probs = model(*(torch.from_numpy(case["feats"][k]).to(dev) for k in cases.FEATURE_KEYS))
        assert np.abs(probs.cpu().numpy() - case["probs"]).max() <= PROB_TOL
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(6):
        model.load_state_dict({k: torch.from_numpy(v) for k, v in b["params"].items()})
        model(*(torch.from_numpy(b["feats"][k]).to(dev) for k in cases.FEATURE_KEYS))
    torch.cuda.synchronize()
    assert free0 - torch.cuda.mem_get_info()[0] < 64 << 20          # no arena piles up


def test_fp16_ragged_batches_and_chunking():
    case = cases.load_case("both_13_16_s2")
    for n, mb in ((1, 4096), (127, 4096), (129, 4096), (1000, 256)):
        sub = cases.slice_case(case, n)
        logits, probs, labels, _ = run_case(sub, "fp16", max_batch=mb)
        check(sub, logits, probs, labels, PROB_TOL, 1.0 - 1.5 / n)              # at most one flip at any of these sizes


def test_ragged_and_tiny_batches_fp32():
    case = cases.load_case("both_small_odd")
    for n in (1, 2, 17, 255):
        sub = cases.slice_case(case, n)
        logits, probs, labels, _ = run_case(sub, "fp32", max_batch=64)   # 255 > 64: internal chunking
        check(sub, logits, probs, labels, FP32_TOL, 1.0)


def test_empty_batch():
    case = cases.load_case("both_small_odd")
    model = case["model"].cuda(0)
    z = torch.zeros(0, 5, device="cuda:0")
    logits, probs = model(z, z, z, z, torch.zeros(0, 5, 8, device="cuda:0"))
    assert tuple(logits.shape) == (0, 2) and tuple(probs.shape) == (0, 2)


def test_cpu_tensor_is_refused_on_gpu_box():
    case = cases.load_case("both_small_odd")
    model = case["model"].cuda(0)
    z = torch.zeros(2, 5)
    with pytest.raises(RuntimeError, match="no CPU path"):
        model(z, z, z, z, torch.zeros(2, 5, 8))


def test_philox_states_are_standard_normal_and_fresh():
    # models.py:169-176 draws new N(0,1) states per call: two calls differ, and the spread
    # of outputs matches what explicit randn states give.
    case = cases.slice_case(cases.load_case("both_13_16_s1234"), 2048)
    dev = torch.device("cuda:0")
    model = cases.build_model(case["entry"], precision="fp32").cuda(0)
    args = [torch.from_numpy(case["feats"][k]).to(dev) for k in cases.FEATURE_KEYS]
    p1 = model(*args)[1].cpu().numpy()
    p2 = model(*args)[1].cpu().numpy()
    d = np.abs(p1 - p2).max()
    assert 1e-4 < d < 0.1            # reference: up to 1.35e-2 between two forwards (SURVEY.md fact 2)
    assert abs(p1[:, 1].mean() - case["probs"][:, 1].mean()) < 2e-3
    assert abs(p1[:, 1].std() - case["probs"][:, 1].std()) < 1e-3


def test_fp16_in_kernel_philox_states():
    # tcgen05 path draws the states inside the layer kernels: fresh per call, N(0,1)-like effect
    case = cases.slice_case(cases.load_case("both_13_16_s1234"), 4096)
    dev = torch.device("cuda:0")
    model = cases.build_model(case["entry"], precision="fp16").cuda(0)
    args = [torch.from_numpy(case["feats"][k]).to(dev) for k in cases.FEATURE_KEYS]
    p1 = model(*args)[1].cpu().numpy()
    p2 = model(*args)[1].cpu().numpy()
    assert np.isfinite(p1).all()
    d = np.abs(p1 - p2).max()
    assert 1e-4 < d < 0.1
    assert abs(p1[:, 1].mean() - case["probs"][:, 1].mean()) < 2e-3
    assert abs(p1[:, 1].std() - case["probs"][:, 1].std()) < 1e-3
    # same site at two different positions of the batch gets different states
    args2 = [a.roll(1, 0) for a in args]
    p3 = model(*args2)[1].cpu().numpy()
    assert np.abs(np.roll(p3, -1, 0) - p1).max() > 1e-4


def test_init_hidden_mode_reproduces_reference_rng_stream():
    # state_mode="init_hidden" draws torch.randn on the CPU generator in the reference's order,
    # so seeding alone reproduces the reference's _call_mods run (same batching).
    e = cases.MANIFEST["callmods"]
    n, bs = e["n"], e["batch"]
    feats = synthetic.make_features(n, 13, 16, seed=e["feature_seed"])
    info = synthetic.make_sampleinfo(n, seed=e["feature_seed"])
    torch.manual_seed(e["weight_seed"])
    from deepsignal_plant_b200.models import ModelBiLSTM
    model = ModelBiLSTM(13, 16, 3, 1, 2, 0, 256, 16, 4, True, True, module="both_bilstm", precision="fp32",
                        state_mode="init_hidden").cuda(0).eval()
    batch = (info, feats["kmer"].astype(np.int64).tolist(), feats["base_means"].tolist(), feats["base_stds"].tolist(),
             feats["base_signal_lens"].astype(np.int64).tolist(), feats["signals"].tolist(), [0] * n)
    torch.manual_seed(e["rng_seed"])
    lines, acc, nb = cm._call_mods(batch, model, bs, 0)
    gold = cases.read_gz("callmods_%d.tsv.gz" % e["rng_seed"]).splitlines()
    assert nb == (n + bs - 1) // bs and len(lines) == len(gold)
    same_label = 0
    for a, b in zip(lines, gold):
        wa, wb = a.split("\t"), b.split("\t")
        assert wa[:6] == wb[:6] and wa[9] == wb[9]
        assert abs(float(wa[6]) - float(wb[6])) <= 2e-6 and abs(float(wa[7]) - float(wb[7])) <= 2e-6
        same_label += wa[8] == wb[8]
    assert same_label / len(gold) >= LABEL_AGREEMENT


def _compare_call_lines(lines, gold, prob_tol):
    """call_mods lines against the reference's: sample info and 5-mer identical, probabilities within prob_tol.
    Returns the number of label flips."""
    assert len(lines) == len(gold)
    flips = 0
    for a, b in zip(lines, gold):
        wa, wb = a.split("\t"), b.split("\t")
        assert len(wa) == 10 and wa[:6] == wb[:6] and wa[9] == wb[9]
        assert abs(float(wa[6]) - float(wb[6])) <= prob_tol and abs(float(wa[7]) - float(wb[7])) <= prob_tol
        flips += wa[8] != wb[8]
    return flips


def test_call_mods_fp16_reproduces_reference_lines():
    # the fp16 path through _call_mods against the reference's own run (callmods_77.tsv.gz), equal seeds
    from oracle.run_ref_callmods import features_batch
    from deepsignal_plant_b200.models import ModelBiLSTM
    e = cases.MANIFEST["callmods"]
    torch.manual_seed(e["weight_seed"])
    model = ModelBiLSTM(13, 16, 3, 1, 2, 0, 256, 16, 4, True, True, module="both_bilstm", precision="fp16",
                        state_mode="init_hidden").cuda(0).eval()
    batch = features_batch(e["n"], 13, 16, e["feature_seed"])
    torch.manual_seed(e["rng_seed"])
    lines, acc, nb = cm._call_mods(batch, model, e["batch"], 0)
    assert model.launch_count() > 0 and nb == (e["n"] + e["batch"] - 1) // e["batch"]
    gold = cases.read_gz("callmods_%d.tsv.gz" % e["rng_seed"]).splitlines()
    assert _compare_call_lines(lines, gold, PROB_TOL) <= max(1, int(len(gold) * (1 - LABEL_AGREEMENT)))


def test_call_mods_worker_loop_reproduces_reference_lines(tmp_path, monkeypatch):
    # _call_mods_q (call_modifications.py:195-259): constructor call with the reference's positional arguments,
    # checkpoint load, queue loop until "kill"; the expectation is the reference's CPU _call_mods run at the same
    # seeds (callmods_99.tsv.gz, manifest "callmods_worker")
    import queue
    import types
    from oracle.run_ref_callmods import features_batch
    from deepsignal_plant_b200.models import ModelBiLSTM
    e = cases.MANIFEST["callmods_worker"]
    n, bs = e["n"], e["batch"]
    torch.manual_seed(e["weight_seed"])
    ckpt = str(tmp_path / "both_bilstm.b13_s16_epoch0.ckpt")
    torch.save(ModelBiLSTM(13, 16, 3, 1, 2, 0, 256, 16, 4, True, True).state_dict(), ckpt)   # train.py:161

    class InitHiddenModel(ModelBiLSTM):
        def __init__(self, *a, **kw):
            super().__init__(*a, state_mode="init_hidden", **kw)
    args = types.SimpleNamespace(seq_len=13, signal_len=16, layernum1=3, layernum2=1, class_num=2, dropout_rate=0, hid_rnn=256,
                                 n_vocab=16, n_embed=4, is_base="yes", is_signallen="yes", model_type="both_bilstm", batch_size=bs)
    fq, pq = queue.Queue(), queue.Queue()
    fq.put(features_batch(n, 13, 16, e["feature_seed"]))
    fq.put("kill")
    orig = cm._call_mods

    def seeded(batch, model, batch_size, device=0):      # the reference run seeds right before _call_mods
        torch.manual_seed(e["rng_seed"])
        return orig(batch, model, batch_size, device)
    monkeypatch.setattr(cm, "ModelBiLSTM", InitHiddenModel)
    monkeypatch.setattr(cm, "_call_mods", seeded)
    cm._call_mods_q(ckpt, fq, pq, None, args, 0)
    lines = pq.get_nowait()
    gold = cases.read_gz("callmods_%d.tsv.gz" % e["rng_seed"]).splitlines()
    assert _compare_call_lines(lines, gold, PROB_TOL) <= 1


def test_forward_host_matches_device_path():
    case = cases.slice_case(cases.load_case("both_13_16_s1"), 3000)
    dev = torch.device("cuda:0")
    model = cases.build_model(case["entry"], precision="fp32", max_batch=1024).cuda(0)
    f = case["feats"]
    logits, probs, labels = model.forward_host(*(f[k] for k in cases.FEATURE_KEYS))
    # Philox states: compare distribution-level agreement with the golden (explicit states)
    assert np.isfinite(probs).all() and probs.shape == (3000, 2)
    assert np.abs(probs - case["probs"]).max() < 0.05
    assert (labels == probs.argmax(1)).all()
    np.testing.assert_allclose(probs.sum(1), 1.0, atol=1e-5)


def test_streaming_host_api_pipelines_batches():
    # submit_host / wait_host: pinned buffers in and out, several batches in flight, chunked staging
    case = cases.slice_case(cases.load_case("both_13_16_s2"), 5000)
    model = cases.build_model(case["entry"], precision="fp16", max_batch=2048).cuda(0)
    f = case["feats"]
    ins = [torch.from_numpy(f[k]).pin_memory() for k in cases.FEATURE_KEYS]
    outs = [(torch.empty((5000, 2)).pin_memory(), torch.empty((5000, 2)).pin_memory(),
             torch.empty((5000,), dtype=torch.int32).pin_memory()) for _ in range(3)]
    tickets = [model.submit_host(*ins, *o) for o in outs]
    for t in reversed(tickets):
        model.wait_host(t)
    for logits, probs, labels in outs:
        p = probs.numpy()
        assert np.isfinite(p).all() and np.abs(p - case["probs"]).max() < 0.05      # Philox states, not the golden ones
        assert (labels.numpy() == p.argmax(1)).all()
        np.testing.assert_allclose(p.sum(1), 1.0, atol=1e-5)
    assert np.abs(outs[0][1].numpy() - outs[1][1].numpy()).max() > 1e-5            # fresh states per submission
    with pytest.raises(ValueError, match="page-locked"):
        model.submit_host(*(torch.from_numpy(f[k]) for k in cases.FEATURE_KEYS), *outs[0])


def test_forward_host_pageable_and_ragged_chunks_fp16():
    case = cases.slice_case(cases.load_case("both_13_16_s1"), 4500)
    model = cases.build_model(case["entry"], precision="fp16", max_batch=1024).cuda(0)     # 5 staged chunks, last ragged
    f = case["feats"]
    logits, probs, labels = model.forward_host(*(f[k] for k in cases.FEATURE_KEYS))
    assert np.isfinite(probs).all() and np.abs(probs - case["probs"]).max() < 0.05
    assert (labels == probs.argmax(1)).all()


@pytest.mark.parametrize("kw", [dict(num_classes=3, is_signallen=False), dict(is_base=False, num_layers1=2, num_layers2=2),
                                dict(module="signal_bilstm", signal_len=32, seq_len=9)])
def test_fp16_unusual_configurations_against_oracle(kw):
    # shapes no fixture covers, on the tensor-core path: 3 classes, no signal-length / no base features,
    # 2-layer branches (second branch layer has K = 256), long signal rows
    a = dict(seq_len=13, signal_len=16, num_layers1=3, num_layers2=1, num_classes=2, hidden_size=256, vocab_size=16,
             embedding_size=4, is_base=True, is_signallen=True, module="both_bilstm")
    a.update(kw)
    cfg = model_oracle.make_cfg(**a)
    torch.manual_seed(17)
    from deepsignal_plant_b200.models import ModelBiLSTM
    model = ModelBiLSTM(a["seq_len"], a["signal_len"], a["num_layers1"], a["num_layers2"], a["num_classes"], 0, 256, 16, 4,
                        a["is_base"], a["is_signallen"], module=a["module"], precision="fp16").cuda(0).eval()
    n = 1111
    feats = synthetic.make_features(n, a["seq_len"], a["signal_len"], seed=17)
    states = synthetic.make_states(cfg, n, seed=18)
    params = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    want = model_oracle.forward(params, cfg, *(feats[k] for k in cases.FEATURE_KEYS), states)[1]
    cases.inject_states(model, states, torch.device("cuda:0"))
    probs = model(*(torch.from_numpy(feats[k]).cuda(0) for k in cases.FEATURE_KEYS))[1].cpu().numpy()
    assert probs.shape == want.shape and np.abs(probs - want).max() <= PROB_TOL
    assert int((probs.argmax(1) != want.argmax(1)).sum()) <= 1                   # 1 111 sites: at most one flip
    assert (model.last_labels.cpu().numpy() == probs.argmax(1)).all()


def test_oracle_agrees_on_fresh_seed():
    # a case that is NOT in the fixtures: oracle and CUDA path on the same seeded inputs
    cfg = model_oracle.make_cfg(seq_len=11, signal_len=10, hidden_size=48, num_layers1=2)
    torch.manual_seed(99)
    from deepsignal_plant_b200.models import ModelBiLSTM
    model = ModelBiLSTM(11, 10, 2, 1, 2, 0, 48, 16, 4, True, True, precision="fp32").cuda(0).eval()
    n = 333
    feats = synthetic.make_features(n, 11, 10, seed=99)
    states = synthetic.make_states(cfg, n, seed=99)
    params = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    want_logits, want_probs = model_oracle.forward(params, cfg, *(feats[k] for k in cases.FEATURE_KEYS), states)
    cases.inject_states(model, states, torch.device("cuda:0"))
    logits, probs = model(*(torch.from_numpy(feats[k]).cuda(0) for k in cases.FEATURE_KEYS))
    assert np.abs(probs.cpu().numpy() - want_probs).max() < FP32_TOL


@pytest.mark.parametrize("which", [0, 1, 2, 3])
def test_tcgen05_building_blocks(which):
    import ctypes as C
    from deepsignal_plant_b200 import _native
    err = C.c_double()
    _native.check(_native.lib().dsp_selftest(0, which, C.byref(err)), "dsp_selftest")
    assert 0 <= err.value < 1e-3, err.value


def test_fp16_scalar_features_outside_the_fp16_range():
    # base_signal_lens are raw sample counts (call_modifications.py:161): a stalled pore gives thousands.  FP16
    # holds integers exactly only to 2 048 and overflows at 65 504; the seq image carries every scalar feature as
    # FP16 value + FP16 residual (lens pre-scaled by 2^-5), so the fp32 reference is matched on such inputs too.
    case = cases.slice_case(cases.load_case("both_13_16_s1"), 1024)
    feats = {k: v.copy() for k, v in case["feats"].items()}
    rng = np.random.default_rng(3)
    lens = feats["base_signal_lens"]
    for value in (2049.0, 4097.0, 70000.0, 1.0e6):
        r, c = rng.integers(0, lens.shape[0], 64), rng.integers(0, lens.shape[1], 64)
        lens[r, c] = value
    feats["base_means"][rng.integers(0, 1024, 32), rng.integers(0, 13, 32)] = 3000.25      # means / stds far off too
    feats["base_stds"][rng.integers(0, 1024, 32), rng.integers(0, 13, 32)] = 70000.0
    feats["signals"][rng.integers(0, 1024, 16), rng.integers(0, 13, 16), 0] = 1.0e5          # clamped, not inf
    want = model_oracle.forward(case["params"], case["cfg"], *(feats[k] for k in cases.FEATURE_KEYS), case["states"])[1]
    dev = torch.device("cuda:0")
    model = cases.build_model(case["entry"], precision="fp16").cuda(0)
    cases.inject_states(model, case["states"], dev)
    probs = model(*(torch.from_numpy(feats[k]).to(dev) for k in cases.FEATURE_KEYS))[1].cpu().numpy()
    assert np.isfinite(probs).all()
    touched = (feats["signals"] > 6.0e4).any(axis=(1, 2))      # the fp32 reference sees 1e5 there, FP16 clamps at 65 504
    err = np.abs(probs - want)[~touched].max()
    agree = (probs.argmax(1) == want.argmax(1))[~touched].mean()
    print("out-of-range scalars: max|dprob|=%.2e agreement=%.5f" % (err, agree))
    assert err <= PROB_TOL and int((probs.argmax(1) != want.argmax(1))[~touched].sum()) <= 1


@pytest.mark.parametrize("seed", [11, 12, 13])
def test_fp16_label_bar_on_100k_sites_per_seed(seed):
    # north_star: labels >= 99.99 % identical.  Random-init prob_1 sits at 0.5 +- 0.003, so the bar needs volume:
    # 102 400 sites per weight seed against the reference forward on torch's CPU operators (oracle/torch_oracle.py,
    # pinned by the same fixtures as the numpy oracle), flips counted and printed.
    from oracle import torch_oracle
    n = 102400
    cfg = model_oracle.make_cfg()
    entry = dict(cases.MANIFEST["forward"]["both_13_16_s1234"])
    entry["weight_seed"] = seed
    dev = torch.device("cuda:0")
    model = cases.build_model(entry, precision="fp16", max_batch=n).cuda(0)
    feats = synthetic.make_features(n, 13, 16, seed=1000 + seed)
    states = synthetic.make_states(cfg, n, seed=2000 + seed)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    torch.set_num_threads(max(1, (os.cpu_count() or 1)))
    want = np.empty((n, 2), np.float32)
    for s in range(0, n, 4096):                              # the oracle in slices (oneDNN workspace), states sliced alike
        e = min(n, s + 4096)
        st = {g: tuple(torch.from_numpy(np.ascontiguousarray(x[:, s:e])) for x in hc) for g, hc in states.items()}
        want[s:e] = torch_oracle.forward(sd, cfg, *(torch.from_numpy(feats[k][s:e]) for k in cases.FEATURE_KEYS), st)[1].numpy()
    cases.inject_states(model, states, dev)
    probs = model(*(torch.from_numpy(feats[k]).to(dev) for k in cases.FEATURE_KEYS))[1].cpu().numpy()
    err = np.abs(probs - want).max()
    flips = int((probs.argmax(1) != want.argmax(1)).sum())
    margin = np.abs(want[:, 1] - 0.5)[probs.argmax(1) != want.argmax(1)]
    print("seed %d: %d sites, max|dprob|=%.2e, %d label flips (%.4f %% identical), largest |p-0.5| of a flipped site %.1e"
          % (seed, n, err, flips, 100.0 * (1 - flips / n), margin.max() if flips else 0.0))
    assert err <= PROB_TOL
    assert flips <= n // 10000, "label agreement %.5f below 99.99 %%" % (1 - flips / n)


def test_exact_epilogue_variant_build_still_matches_reference():
    # the shipped library evaluates the gate non-linearities with tanh.approx (DSP_TANH_APPROX=2); the 2^x + reciprocal
    # epilogue (-DDSP_TANH_APPROX=0, ~1e-7 relative error) stays buildable as libdsp_b200_exact.so:
    #   DSP_B200_VARIANT=exact DSP_B200_DEFINES=-DDSP_TANH_APPROX=0 python -m deepsignal_plant_b200.build
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib = os.path.join(root, "deepsignal_plant_b200", "libdsp_b200_exact.so")
    if not os.path.exists(lib):
        pytest.skip("variant build libdsp_b200_exact.so is not present")
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import numpy as np, torch, cases\n"
            "case = cases.slice_case(cases.load_case('both_13_16_s2'), 4096)\n"
            "m = cases.build_model(case['entry'], precision='fp16').cuda(0)\n"
            "cases.inject_states(m, case['states'], torch.device('cuda:0'))\n"
            "p = m(*(torch.from_numpy(case['feats'][k]).cuda(0) for k in cases.FEATURE_KEYS))[1].cpu().numpy()\n"
            "print('ERR %%.3e AGREE %%.5f' %% (np.abs(p - case['probs']).max(), (p.argmax(1) == case['probs'].argmax(1)).mean()))\n"
            % (root, os.path.join(root, "tests")))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, env=dict(os.environ, DSP_B200_LIB=lib))
    assert r.returncode == 0, r.stderr[-2000:]
    err, agree = [l for l in r.stdout.splitlines() if l.startswith("ERR")][-1].split()[1::2]
    assert float(err) <= PROB_TOL and float(agree) >= LABEL_AGREEMENT
