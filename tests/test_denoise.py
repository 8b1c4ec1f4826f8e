"""``denoise``: the flags, the round halves, the cleaning rule and the writers (CPU), the reference's own
``clean_samples`` where the reference is built, and the command end to end on a separable set with flipped labels
(GPU)."""
import os

import numpy as np
import pytest
import torch

from deepsignal_plant_b200 import cli, synthetic
from deepsignal_plant_b200 import denoise as dn
from deepsignal_plant_b200 import train as tr

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


def write_set(tmp_path, f, labels, name="set"):
    """The labelled sites as a text feature file and as a .dspf file."""
    from deepsignal_plant_b200.feature_bin import pack_feature_file
    from deepsignal_plant_b200.feature_io import features_to_str
    f = dict(f)
    f["base_means"] = np.round(f["base_means"].astype(np.float64), 6).astype(np.float32)
    txt = tmp_path / (name + ".tsv")
    with open(txt, "w") as fh:
        for i in range(len(labels)):
            info = "chr1\t%d\t+\t%d\tread%d\tt" % (1000 + i, 1000 + i, i)
            fh.write(features_to_str(info, f["kmer"][i], f["base_means"][i], f["base_stds"][i], f["base_signal_lens"][i],
                                     f["signals"][i], labels[i]) + "\n")
    binp = tmp_path / (name + ".dspf")
    pack_feature_file(str(txt), str(binp))
    return str(txt), str(binp)


def flipped_set(n, seed, frac=0.15):
    """A separable set in which ``frac`` of the label-0 sites are relabelled 1 -> (features, noisy labels, flipped)."""
    f, labels = labelled_features(n, seed=seed)
    rng = np.random.default_rng(seed + 2)
    neg = np.nonzero(labels == 0)[0]
    flip = np.sort(rng.choice(neg, int(frac * neg.size), replace=False))
    noisy = labels.copy()
    noisy[flip] = 1
    return f, noisy, labels, flip


def denoise_args(*extra):
    return cli.build_parser().parse_args(["denoise", "--train_file", "t"] + list(extra))


# ---- CPU -------------------------------------------------------------------------------------------------------
def test_denoise_flags_parse_with_reference_defaults():
    a = denoise_args()
    want = dict(train_file="t", is_filter_fn="no", model_type="signal_bilstm", seq_len=13, signal_len=16, layernum1=3,
                layernum2=1, class_num=2, dropout_rate=0.5, n_vocab=16, n_embed=4, is_base="yes", is_signallen="yes",
                hid_rnn=256, pos_weight=1.0, batch_size=512, lr=0.001, epoch_num=3, step_interval=100, iterations=10,
                rounds=3, score_cf=0.5, kept_ratio=0.99, tseed=1234)
    for k, v in want.items():
        assert getattr(a, k) == v, k
    with pytest.raises(SystemExit):
        cli.build_parser().parse_args(["denoise"])


def test_denoise_subcommand_dispatches(monkeypatch):
    seen = []
    monkeypatch.setattr(dn, "main", lambda args: seen.append(args))
    assert cli.main(["denoise", "--train_file", "x.tsv", "--rounds", "2"]) == 0
    assert len(seen) == 1 and seen[0].train_file == "x.tsv" and seen[0].rounds == 2


@pytest.mark.parametrize("n", [2, 3, 10, 11, 1001])
def test_round_halves_partition_the_set(n):
    for r in range(3):
        a, b = dn.round_halves(n, 1234, 0, r)
        assert a.numel() == n // 2 and b.numel() == n - n // 2
        assert torch.equal(torch.sort(torch.cat([a, b])).values, torch.arange(n))
        a2, b2 = dn.round_halves(n, 1234, 0, r)
        assert torch.equal(a, a2) and torch.equal(b, b2)
    if n > 10:
        assert not torch.equal(dn.round_halves(n, 1234, 0, 0)[0], dn.round_halves(n, 1234, 0, 1)[0])
        assert not torch.equal(dn.round_halves(n, 1234, 0, 0)[0], dn.round_halves(n, 1234, 1, 0)[0])
        assert not torch.equal(dn.round_halves(n, 1234, 0, 0)[0], dn.round_halves(n, 99, 0, 0)[0])


def test_model_seeds_are_distinct_and_fixed():
    seeds = {dn.model_seed(1234, k, r, h) for k in range(10) for r in range(3) for h in range(3)}
    assert len(seeds) == 90 and all(0 <= s < 2 ** 40 for s in seeds)
    assert dn.model_seed(1234, 0, 0, 0) == dn.model_seed(1234, 0, 0, 0) != dn.model_seed(1235, 0, 0, 0)


def test_mean_is_float64_in_round_order():
    s = np.array([[1.0, 0.1], [1e-8, 0.2], [1e-8, 0.3]], np.float32)
    mean, std = dn.score_stats(s)
    acc = np.float64(np.float32(1.0)) + np.float64(np.float32(1e-8)) + np.float64(np.float32(1e-8))
    assert mean[0] == acc / 3
    rows = s.astype(np.float64)
    want = ((rows[0] + rows[1]) + rows[2]) / 3
    assert np.array_equal(mean, want)
    assert np.allclose(std, rows.std(0), rtol=0, atol=1e-15)
    assert mean.dtype == np.float64


def test_cleaning_rule_keeps_a_mean_equal_to_the_cutoff():
    labels = np.array([1, 1, 1, 0, 0, 0])
    mean = np.array([0.5, 0.4999999, 0.9, 0.5, 0.9, 0.1])
    keep, c = dn.clean(labels, mean, 0.5, False)
    assert keep.tolist() == [True, False, True, True, True, True]
    assert (c["positives"], c["negatives"], c["kept_positives"], c["kept_negatives"]) == (3, 3, 2, 3)
    assert c["left_ratio"] == 2 / 3 and c["left_ratio2"] == 1.0
    keep, c = dn.clean(labels, mean, 0.5, True)
    assert keep.tolist() == [True, False, True, True, False, True]
    assert c["left_ratio2"] == 2 / 3
    # the float32 scores 0.25, 0.75 average to exactly 0.5 in float64
    m, _ = dn.score_stats(np.array([[0.25], [0.75]], np.float32))
    assert dn.clean(np.array([1]), m, 0.5, False)[0].tolist() == [True]


def test_stop_rule():
    assert dn.should_stop(dict(left_ratio=0.99, left_ratio2=1.0), 0.99)
    assert not dn.should_stop(dict(left_ratio=0.98, left_ratio2=1.0), 0.99)
    assert not dn.should_stop(dict(left_ratio=1.0, left_ratio2=0.98), 0.99)


def test_output_names():
    assert dn.output_path("/d/samples.tsv", 1, False) == "/d/samples.denoise_fp1.tsv"
    assert dn.output_path("/d/samples.tsv", 3, True) == "/d/samples.denoise_fnp3.tsv"
    assert dn.output_path("/d/s.dspf", 2, False) == "/d/s.denoise_fp2.dspf"


def test_text_writer_keeps_lines_byte_for_byte(tmp_path):
    f, labels = labelled_features(50, seed=3)
    txt, _ = write_set(tmp_path, f, labels)
    rows = np.array([0, 3, 4, 17, 49])
    out = str(tmp_path / "out.tsv")
    dn.write_kept(txt, out, rows)
    lines = open(txt, "rb").readlines()
    assert open(out, "rb").read() == b"".join(lines[i] for i in rows)


def test_dspf_writer_keeps_rows_bit_for_bit(tmp_path):
    from deepsignal_plant_b200.feature_bin import FeatureBinReader
    f, labels = labelled_features(70, seed=4)
    _, binp = write_set(tmp_path, f, labels)
    rows = np.array([1, 2, 30, 31, 69])
    out = str(tmp_path / "out.dspf")
    dn.write_kept(binp, out, rows)

    def read(path):
        parts = {k: [] for k in KEYS + ("labels", "info")}
        for b in FeatureBinReader(path, pinned=False, slots=2):
            for k, t in zip(KEYS + ("labels",), b.arrays() + (b.labels,)):
                parts[k].append(t[:b.n].numpy().copy())
            off = b.info_off[:b.n + 1]
            parts["info"] += [bytes(b.info_text[off[i]:off[i + 1]]) for i in range(b.n)]
        return {k: (v if k == "info" else np.concatenate(v)) for k, v in parts.items()}
    a, b = read(binp), read(out)
    for k in KEYS + ("labels",):
        assert a[k][rows].tobytes() == b[k].tobytes(), k
    assert [a["info"][i] for i in rows] == b["info"]


def test_refusals(tmp_path):
    gz = tmp_path / "s.tsv.gz"
    gz.write_bytes(b"")
    with pytest.raises(ValueError, match="decompress"):
        dn.denoise(_with(denoise_args(), train_file=str(gz)))
    empty = tmp_path / "empty.tsv"
    empty.write_text("")
    with pytest.raises(ValueError):
        dn.denoise(_with(denoise_args(), train_file=str(empty)))
    f, labels = labelled_features(20, seed=5)
    txt, _ = write_set(tmp_path, f, np.zeros_like(labels), name="neg")
    with pytest.raises(ValueError, match="no label-1"):
        dn.denoise(_with(denoise_args(), train_file=txt))
    one, _ = write_set(tmp_path, {k: v[:1] for k, v in f.items()}, np.ones(1, np.int32), name="one")
    with pytest.raises(ValueError, match="at least 2"):
        dn.denoise(_with(denoise_args(), train_file=one))
    with pytest.raises(ValueError, match="at least 1"):
        dn.denoise(_with(denoise_args(), train_file=txt, rounds=0))
    with pytest.raises(ValueError, match="at least 1"):
        dn.denoise(_with(denoise_args(), train_file=txt, iterations=0))


def test_refused_under_torchrun(monkeypatch):
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(RuntimeError, match="multi-GPU denoise is not supported"):
        dn.denoise(denoise_args())


def _with(args, **kw):
    for k, v in kw.items():
        setattr(args, k, v)
    return args


def test_reference_clean_samples_writes_the_same_file(tmp_path):
    from oracle import ref_import
    if not ref_import.available():
        pytest.skip("the reference is not built (oracle/_ref)")
    ref = ref_import.import_reference("denoise")
    f, labels = labelled_features(60, seed=6)
    txt, _ = write_set(tmp_path, f, labels)
    scores = np.random.default_rng(1).random((3, 60)).astype(np.float32)
    mean, _ = dn.score_stats(scores)
    keep, _ = dn.clean(labels, mean, 0.5, False)
    ours = str(tmp_path / "ours.tsv")
    dn.write_kept(txt, ours, np.nonzero(keep)[0])
    # the reference keys a sample's scores by its line index and lists them in round order; clean_samples writes the
    # kept lines next to its input and returns that path (first in a tuple, with the kept ratios after it)
    idx2scores = {i: [float(s) for s in scores[:, i]] for i in range(60)}
    res = ref.clean_samples(txt, idx2scores, 0.5, False)
    theirs = res[0] if isinstance(res, tuple) else res
    assert open(theirs, "rb").read() == open(ours, "rb").read()


# ---- GPU: end to end ---------------------------------------------------------------------------------------------
# Thresholds set from the first B200 run with margin; the observed values are recorded in DESIGN §9.
MIN_FLIPPED_REMOVED = 0.70
MIN_TRUE_POSITIVES_KEPT = 0.90

SMALL = ["--hid_rnn", "32", "--iterations", "2", "--rounds", "2", "--epoch_num", "2", "--batch_size", "64",
         "--lr", "0.005", "--kept_ratio", "1.0"]


@pytest.mark.gpu
def test_denoise_end_to_end(tmp_path):
    n = 8001
    f, noisy, clean_labels, flip = flipped_set(n, seed=31)
    txt, binp = write_set(tmp_path, f, noisy)
    res = dn.denoise(cli.build_parser().parse_args(["denoise", "--train_file", txt] + SMALL))
    print("denoise end to end, per iteration:", res["iterations"])
    assert len(res["iterations"]) == 2
    assert res["path"] == dn.output_path(txt, 2, False) and os.path.exists(res["path"])
    assert not os.path.exists(dn.output_path(txt, 1, False)) and os.path.exists(txt)
    kept = res["samples"][-1][dn.clean(noisy[res["samples"][-1]], dn.score_stats(res["scores"][-1])[0], 0.5, False)[0]]
    true_pos = np.nonzero(clean_labels == 1)[0]
    removed_flipped = 1.0 - np.isin(flip, kept).mean()
    kept_true = np.isin(true_pos, kept).mean()
    print("denoise end to end: %d sites, %d flipped; removed %.4f of the flipped, kept %.4f of the true positives; %s"
          % (n, flip.size, removed_flipped, kept_true, res["iterations"]))
    assert removed_flipped >= MIN_FLIPPED_REMOVED
    assert kept_true >= MIN_TRUE_POSITIVES_KEPT
    assert np.isin(np.nonzero(noisy == 0)[0], kept).all()
    lines = open(txt, "rb").readlines()
    first = open(res["path"], "rb").read()
    assert first == b"".join(lines[i] for i in kept)
    # a second run: the same file; max_models=1: the same scores
    res2 = dn.denoise(cli.build_parser().parse_args(["denoise", "--train_file", txt] + SMALL), max_models=1)
    assert open(res2["path"], "rb").read() == first
    for a, b in zip(res["scores"], res2["scores"]):
        assert a.tobytes() == b.tobytes()
    res3 = dn.denoise(cli.build_parser().parse_args(["denoise", "--train_file", txt] + SMALL))
    assert open(res3["path"], "rb").read() == first
    # the .dspf input keeps the same samples
    resb = dn.denoise(cli.build_parser().parse_args(["denoise", "--train_file", binp] + SMALL))
    assert resb["path"] == dn.output_path(binp, 2, False)
    assert np.array_equal(resb["samples"][-1], res["samples"][-1])
    got = tr.load_feature_set(resb["path"], 13, 16)
    src = tr.load_feature_set(binp, 13, 16)
    for k in KEYS + ("labels",):
        assert torch.equal(got[k], src[k][torch.from_numpy(kept)]), k


@pytest.mark.gpu
def test_denoised_file_trains_and_calls(tmp_path):
    f, noisy, _, _ = flipped_set(3000, seed=41)
    txt, _ = write_set(tmp_path, f, noisy)
    assert cli.main(["denoise", "--train_file", txt, "--model_type", "both_bilstm"] + SMALL[:2] +
                    ["--iterations", "1", "--rounds", "1", "--epoch_num", "1", "--batch_size", "128"]) == 0
    cleaned = dn.output_path(txt, 1, False)
    fv, lv = labelled_features(1024, seed=42)
    _, va = write_set(tmp_path, fv, lv, name="valid")
    mdir = tmp_path / "models"
    assert cli.main(["train", "--train_file", cleaned, "--valid_file", va, "--model_dir", str(mdir), "--hid_rnn", "32",
                     "--max_epoch_num", "1", "--min_epoch_num", "1", "--batch_size", "128"]) == 0
    ckpt = sorted(os.listdir(mdir))[0]
    out = tmp_path / "calls.tsv"
    assert cli.main(["call_mods", "-i", va, "-m", str(mdir / ckpt), "-o", str(out), "--hid_rnn", "32"]) == 0
    assert len(open(out).readlines()) == 1024
