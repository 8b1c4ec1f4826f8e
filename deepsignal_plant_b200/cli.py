"""Command line of the B200 hot path: the ``call_mods`` and ``call_freq`` sub-commands of
``deepsignal_plant`` (``deepsignal_plant/deepsignal_plant.py:106-107,204-316,438-475``) with the
reference's flag names and defaults.

    python -m deepsignal_plant_b200 call_mods -i features.tsv -m model.ckpt -o calls.tsv
    python -m deepsignal_plant_b200 call_freq -i calls.tsv -o freq.tsv [--bed] [--sort]

    python -m deepsignal_plant_b200 extract   -i reads.npz -o features.tsv      # decoded reads -> the reference's feature file
    python -m deepsignal_plant_b200 extract   -i reads.npz -o features.dspf     # ... -> binary hand-off (feature_bin.py)
    python -m deepsignal_plant_b200 call_mods -i features.dspf -m model.ckpt -o calls.tsv      # same calls, no text parsing
    python -m deepsignal_plant_b200 pack_features -i features.tsv -o features.dspf             # an existing text file -> binary
    python -m deepsignal_plant_b200 denoise --train_file samples.tsv      # -> samples.denoise_fp<k>.tsv, then train on it
    python -m deepsignal_plant_b200 train --train_file train.dspf --valid_file valid.dspf --model_dir models/

Multi-GPU: launch ``call_mods``, ``call_freq`` or ``train`` under torchrun, one process per GPU.  ``call_mods`` cuts the
feature file (or the reads archive) into contiguous shards and concatenates the output in file order, no collective on
the data path; ``call_freq`` parses contiguous byte shards, exchanges the records by site key over NVLink peer memory and
every rank writes its slice of the table (freq_dist.py); ``train`` keeps ``--batch_size`` as the global batch, every
rank trains on a slice of each step and the gradients are summed by a deterministic all-reduce over NVLink peer
memory, so the replicas stay bit-identical and rank 0 writes the checkpoints (train_dist.py).  ``extract`` here takes reads that are already decoded
(reading fast5 needs h5py: outside this implementation); ``train`` runs the reference's training loop on the fp32 training kernels (train.py), with
``--optim_type Adam|RMSprop|SGD|Ranger`` (Ranger's step is one fused kernel per parameter group, optim.py); ``denoise``
removes unsupported positive samples before ``train``, training each iteration's cross-validation models together in
model-batched steps (denoise.py).  ``denoise`` runs on one GPU; under torchrun it is refused."""
from __future__ import annotations

import argparse
import sys


def add_train_parser(sub):
    """The reference's ``train`` flags and defaults (``deepsignal_plant.py`` train parser)."""
    tp = sub.add_parser("train", description="train a model on labelled features (.dspf or the reference's text file)")
    g = tp.add_argument_group("INPUT")
    g.add_argument("--train_file", type=str, required=True)
    g.add_argument("--valid_file", type=str, required=True)
    g = tp.add_argument_group("OUTPUT")
    g.add_argument("--model_dir", type=str, required=True)
    g = tp.add_argument_group("MODEL_HYPER")
    g.add_argument("--model_type", type=str, default="both_bilstm",
                   choices=["both_bilstm", "seq_bilstm", "signal_bilstm"], required=False)
    g.add_argument("--seq_len", type=int, default=13, required=False)
    g.add_argument("--signal_len", type=int, default=16, required=False)
    g.add_argument("--layernum1", type=int, default=3, required=False)
    g.add_argument("--layernum2", type=int, default=1, required=False)
    g.add_argument("--class_num", type=int, default=2, required=False)
    g.add_argument("--dropout_rate", type=float, default=0.5, required=False)
    g.add_argument("--n_vocab", type=int, default=16, required=False)
    g.add_argument("--n_embed", type=int, default=4, required=False)
    g.add_argument("--is_base", type=str, default="yes", required=False)
    g.add_argument("--is_signallen", type=str, default="yes", required=False)
    g.add_argument("--hid_rnn", type=int, default=256, required=False)
    g = tp.add_argument_group("TRAINING")
    g.add_argument("--optim_type", type=str, default="Adam", choices=["Adam", "RMSprop", "SGD", "Ranger"],
                   required=False)
    g.add_argument("--batch_size", type=int, default=512, required=False)
    g.add_argument("--lr", type=float, default=0.001, required=False)
    g.add_argument("--max_epoch_num", type=int, default=10, required=False)
    g.add_argument("--min_epoch_num", type=int, default=5, required=False)
    g.add_argument("--step_interval", type=int, default=100, required=False)
    g.add_argument("--pos_weight", type=float, default=1.0, required=False)
    g.add_argument("--init_model", type=str, default=None, required=False)
    g.add_argument("--tseed", type=int, default=1234, required=False)
    return tp


def add_denoise_parser(sub):
    """The reference's ``denoise`` flags and defaults (``deepsignal_plant.py`` denoise parser)."""
    dp = sub.add_parser("denoise", description="remove positive training samples whose label the data does not support "
                                               "(labelled features: .dspf or the reference's text file)")
    g = dp.add_argument_group("INPUT")
    g.add_argument("--train_file", type=str, required=True)
    g = dp.add_argument_group("FILTER")
    g.add_argument("--is_filter_fn", type=str, default="no", required=False,
                   help="also remove negative samples the models score as positive; default no")
    g = dp.add_argument_group("MODEL_HYPER")
    g.add_argument("--model_type", type=str, default="signal_bilstm",
                   choices=["both_bilstm", "seq_bilstm", "signal_bilstm"], required=False)
    g.add_argument("--seq_len", type=int, default=13, required=False)
    g.add_argument("--signal_len", type=int, default=16, required=False)
    g.add_argument("--layernum1", type=int, default=3, required=False)
    g.add_argument("--layernum2", type=int, default=1, required=False)
    g.add_argument("--class_num", type=int, default=2, required=False)
    g.add_argument("--dropout_rate", type=float, default=0.5, required=False)
    g.add_argument("--n_vocab", type=int, default=16, required=False)
    g.add_argument("--n_embed", type=int, default=4, required=False)
    g.add_argument("--is_base", type=str, default="yes", required=False)
    g.add_argument("--is_signallen", type=str, default="yes", required=False)
    g.add_argument("--hid_rnn", type=int, default=256, required=False)
    g = dp.add_argument_group("TRAINING")
    g.add_argument("--pos_weight", type=float, default=1.0, required=False)
    g.add_argument("--batch_size", type=int, default=512, required=False)
    g.add_argument("--lr", type=float, default=0.001, required=False)
    g.add_argument("--epoch_num", type=int, default=3, required=False)
    g.add_argument("--step_interval", type=int, default=100, required=False)
    g = dp.add_argument_group("DENOISE")
    g.add_argument("--iterations", type=int, default=10, required=False)
    g.add_argument("--rounds", type=int, default=3, required=False)
    g.add_argument("--score_cf", type=float, default=0.5, required=False,
                   help="score cutoff to keep a sample; default 0.5")
    g.add_argument("--kept_ratio", type=float, default=0.99, required=False,
                   help="stop once this fraction of the positive (and, with --is_filter_fn, negative) samples is kept")
    g.add_argument("--tseed", type=int, default=1234, required=False)
    return dp


def build_parser():
    parser = argparse.ArgumentParser(prog="deepsignal_plant_b200",
                                     description="deepsignal-plant extract / call_mods / call_freq on B200 (sm_100a) kernels")
    sub = parser.add_subparsers(title="modules", dest="module")
    cm = sub.add_parser("call_mods", description="call modifications")
    cf = sub.add_parser("call_freq", description="call frequency of modifications at genome level")
    add_train_parser(sub)
    add_denoise_parser(sub)

    ex = sub.add_parser("extract", description="extract features from decoded re-squiggled reads (an .npz archive written by "
                                               "extract_features.save_reads) into the reference's feature file")
    g = ex.add_argument_group("INPUT")
    g.add_argument("--fast5_dir", "-i", action="store", type=str, required=True,
                   help="the decoded-reads archive (.npz); the reference's flag name is kept")
    g.add_argument("--recursively", "-r", action="store", type=str, required=False, default="yes",
                   help="accepted for compatibility (the input is one archive of decoded reads, not a directory tree)")
    g.add_argument("--corrected_group", action="store", type=str, required=False, default="RawGenomeCorrected_000",
                   help="accepted for compatibility (used when the archive is made)")
    g.add_argument("--basecall_subgroup", action="store", type=str, required=False, default="BaseCalled_template",
                   help="accepted for compatibility (used when the archive is made)")
    g.add_argument("--is_dna", action="store", type=str, required=False, default="yes")
    g.add_argument("--reference_path", action="store", type=str, required=False, default=None)
    g = ex.add_argument_group("EXTRACTION")
    g.add_argument("--normalize_method", action="store", type=str, choices=["mad", "zscore"], default="mad", required=False)
    g.add_argument("--methy_label", action="store", type=int, choices=[1, 0], required=False, default=1)
    g.add_argument("--seq_len", action="store", type=int, required=False, default=13)
    g.add_argument("--signal_len", action="store", type=int, required=False, default=16)
    g.add_argument("--motifs", action="store", type=str, required=False, default="CG")
    g.add_argument("--mod_loc", action="store", type=int, required=False, default=0)
    g.add_argument("--region", action="store", type=str, required=False, default=None)
    g.add_argument("--positions", action="store", type=str, required=False, default=None)
    g = ex.add_argument_group("OUTPUT")
    g.add_argument("--write_path", "-o", action="store", type=str, required=True,
                   help="the feature file; a name ending in .dspf selects the binary hand-off format that call_mods reads "
                        "without parsing text (feature_bin.py), anything else the reference's 12-column text")
    g.add_argument("--w_is_dir", action="store", type=str, required=False, default="no",
                   help="only 'no' (one output file) is supported")
    g.add_argument("--w_batch_num", action="store", type=int, required=False, default=200, help="accepted for compatibility")
    g.add_argument("--gzip", action="store_true", default=False, required=False)
    ex.add_argument("--nproc", "-p", action="store", type=int, default=10, required=False,
                    help="the reference's number of worker processes: kept with its default; the native formatters use --host_threads")
    ex.add_argument("--host_threads", action="store", type=int, default=0, help="host threads for formatting; 0 = all cores")
    ex.add_argument("--f5_batch_size", action="store", type=int, default=30, required=False, help="reads per extraction chunk")

    pk = sub.add_parser("pack_features", description="convert a text feature file of `extract` (plain or .gz) into the binary "
                                                     "hand-off format that call_mods reads without parsing text (.dspf, feature_bin.py)")
    pk.add_argument("--input_path", "-i", action="store", type=str, required=True, help="the 12-column text feature file")
    pk.add_argument("--write_path", "-o", action="store", type=str, required=True, help="the binary feature file to write")
    pk.add_argument("--host_threads", action="store", type=int, default=0, help="parser threads; 0 = all cores")

    g = cm.add_argument_group("INPUT")
    g.add_argument("--input_path", "-i", action="store", type=str, required=True,
                   help="a signal_feature file from `deepsignal_plant extract` (plain or .gz), a binary feature file (.dspf from "
                        "`extract -o x.dspf` or feature_bin.pack_feature_file), or a decoded-reads archive "
                        "(.npz written by extract_features.save_reads) to extract and call in one pass")
    g.add_argument("--f5_batch_size", action="store", type=int, default=30, required=False,
                   help="reads per extraction chunk for a decoded-reads archive; feature files are cut by site count")
    g = cm.add_argument_group("EXTRACTION (when --input_path is a decoded-reads .npz archive instead of a feature file)")
    g.add_argument("--normalize_method", action="store", type=str, choices=["mad", "zscore"], default="mad", required=False)
    g.add_argument("--motifs", action="store", type=str, required=False, default="CG")
    g.add_argument("--mod_loc", action="store", type=int, required=False, default=0)
    g.add_argument("--is_dna", action="store", type=str, required=False, default="yes")
    g.add_argument("--reference_path", action="store", type=str, required=False, default=None,
                   help="genome FASTA: contig lengths give the pos_in_strand column")
    g.add_argument("--positions", action="store", type=str, required=False, default=None)
    g.add_argument("--region", action="store", type=str, required=False, default=None)
    g.add_argument("--methy_label", action="store", type=int, choices=[1, 0], required=False, default=1,
                   help="accepted for compatibility (the label column is not part of the calls)")
    g.add_argument("--recursively", "-r", action="store", type=str, required=False, default="yes", help="accepted for compatibility")
    g.add_argument("--corrected_group", action="store", type=str, required=False, default="RawGenomeCorrected_000",
                   help="accepted for compatibility (used when the archive is made)")
    g.add_argument("--basecall_subgroup", action="store", type=str, required=False, default="BaseCalled_template",
                   help="accepted for compatibility (used when the archive is made)")
    g = cm.add_argument_group("CALL")
    g.add_argument("--model_path", "-m", action="store", type=str, required=True, help="file path of the trained model (.ckpt)")
    g.add_argument("--model_type", type=str, default="both_bilstm", choices=["both_bilstm", "seq_bilstm", "signal_bilstm"])
    g.add_argument("--seq_len", type=int, default=13)
    g.add_argument("--signal_len", type=int, default=16)
    g.add_argument("--layernum1", type=int, default=3)
    g.add_argument("--layernum2", type=int, default=1)
    g.add_argument("--class_num", type=int, default=2)
    g.add_argument("--dropout_rate", type=float, default=0)
    g.add_argument("--n_vocab", type=int, default=16)
    g.add_argument("--n_embed", type=int, default=4)
    g.add_argument("--is_base", type=str, default="yes")
    g.add_argument("--is_signallen", type=str, default="yes")
    g.add_argument("--batch_size", "-b", default=512, type=int,
                   help="accepted for compatibility; the kernels take whole staged batches (--max_batch)")
    g.add_argument("--hid_rnn", type=int, default=256)
    g.add_argument("--max_batch", type=int, default=65536, help="sites per staged batch (workspace size)")
    g = cm.add_argument_group("OUTPUT")
    g.add_argument("--result_file", "-o", action="store", type=str, required=True)
    g.add_argument("--gzip", action="store_true", default=False)
    g = cm.add_argument_group("CALL_FREQ IN THE SAME RUN (the per-site table without re-reading the calls file; under torchrun the "
                              "ranks exchange their calls over NVLink, see call_freq)")
    g.add_argument("--freq_out", type=str, default=None, help="also write the call_freq table of this run's calls here")
    g.add_argument("--freq_prob_cf", type=float, default=0.5, help="call_freq --prob_cf")
    g.add_argument("--freq_bed", action="store_true", default=False, help="call_freq --bed")
    g.add_argument("--freq_sort", action="store_true", default=False, help="call_freq --sort")
    cm.add_argument("--nproc", "-p", action="store", type=int, default=10,
                    help="the reference's number of worker processes: kept with its default; the native parser / formatter use --host_threads")
    cm.add_argument("--host_threads", action="store", type=int, default=0,
                    help="host threads for parsing / formatting; 0 (default) = all cores, shared evenly between the ranks of a torchrun job")
    cm.add_argument("--reader_threads", action="store", type=int, default=0,
                    help="host threads of the feature reader alone (0 = --host_threads for text, min(8, --host_threads) for .dspf)")
    cm.add_argument("--format_threads", action="store", type=int, default=0,
                    help="host threads of the output formatter alone (0 = min(8, --host_threads))")
    cm.add_argument("--stream_depth", action="store", type=int, default=3,
                    help="feature batches in flight on the device (1-6); the reader keeps this many + 6 page-locked slots")
    cm.add_argument("--nproc_gpu", action="store", type=int, default=2,
                    help="accepted for compatibility; use torchrun for one process per GPU")

    g = cf.add_argument_group("INPUT")
    g.add_argument("--input_path", "-i", action="append", type=str, required=True)
    g.add_argument("--file_uid", type=str, action="store", required=False, default=None)
    g = cf.add_argument_group("OUTPUT")
    g.add_argument("--result_file", "-o", action="store", type=str, required=True)
    g.add_argument("--bed", action="store_true", default=False)
    g.add_argument("--sort", action="store_true", default=False)
    g.add_argument("--gzip", action="store_true", default=False)
    g = cf.add_argument_group("CAlCULATE")
    g.add_argument("--prob_cf", type=float, action="store", required=False, default=0.5)
    g = cf.add_argument_group("PARALLEL")
    g.add_argument("--contigs", action="store", type=str, required=False, default=None,
                   help="a genome FASTA, a file with one contig name per line, or a comma-separated list: only these contigs are "
                        "aggregated, one GPU pass per contig, and the rows come out contig by contig in the order of the reference's "
                        "per-contig mode (call_mods_freq.py:203-215)")
    g.add_argument("--nproc", action="store", type=int, required=False, default=1,
                   help="accepted for compatibility (the reference's per-contig worker processes; here: torchrun ranks)")
    g.add_argument("--max_host_records", action="store", type=int, required=False, default=0,
                   help="records whose parsed columns may sit in host memory at once (80 bytes each; 0 = half of the available "
                        "memory); a larger input is aggregated in key-hash shards, the files re-read once per shard, same table")
    return parser


def _warm_device_while_importing():
    """The CUDA context of this rank's GPU comes up on a side thread (dsp_device_warmup: ctypes only) while the main
    thread imports torch and reads the checkpoint -- about a second of a fresh process's start-up, off the critical path.
    Failures are left to the real call sites, which report them."""
    import os
    import threading

    def warm():
        try:
            from . import _native
            _native.lib().dsp_device_warmup(int(os.environ.get("LOCAL_RANK", "0")))
        except Exception:                                   # noqa: BLE001 -- no GPU / no library: reported by call_mods itself
            pass
    threading.Thread(target=warm, daemon=True).start()


def main(argv=None):
    parser = build_parser()
    args = parser.parse_args(argv)
    if args.module == "call_mods":
        _warm_device_while_importing()
        from .call_modifications import call_mods
        call_mods(args)
    elif args.module == "extract":
        from .extract_features import extract_to_file
        extract_to_file(args)
    elif args.module == "pack_features":
        from .feature_bin import pack_feature_file
        n = pack_feature_file(args.input_path, args.write_path, nthreads=args.host_threads or None)
        print("[pack_features] {} sites -> {}".format(n, args.write_path))
    elif args.module == "train":
        from .train import main as train_main
        train_main(args)
    elif args.module == "denoise":
        from .denoise import main as denoise_main
        denoise_main(args)
    elif args.module == "call_freq":
        from .call_mods_freq import call_mods_frequency_to_file
        call_mods_frequency_to_file(args)
    else:
        parser.print_help()
        return 2
    return 0


if __name__ == "__main__":
    sys.exit(main())
