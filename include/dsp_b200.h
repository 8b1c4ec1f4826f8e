/*
 * dsp_b200.h -- C ABI of libdsp_b200.so, the B200 (sm_100a) implementation of
 * deepsignal-plant's per-site methylation classifier hot path.
 *
 * The reference (PengNi/deepsignal-plant v0.1.6) is pure Python and has no FFI of its
 * own; the boundary it exposes for this path is the torch.nn.Module API of
 * ModelBiLSTM (deepsignal_plant/models.py:99-240) as driven by _call_mods
 * (deepsignal_plant/call_modifications.py:130-192) and, for the optional per-site
 * aggregation, calculate_mods_frequency (deepsignal_plant/call_mods_freq.py:29-74).
 * Each entry point below names the reference interface it stands behind.  The Python
 * mirror of that interface lives in deepsignal_plant_b200/ and binds these symbols
 * with ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions: plain C types only, no torch types.  Every function returns 0 on
 * success and a non-zero dsp_status otherwise; dsp_last_error() returns a
 * thread-local message for the last failure.  No exception crosses the ABI.
 * Unless stated otherwise pointers are DEVICE pointers on the handle's device, the
 * call only enqueues work on `stream` (a cudaStream_t passed as void*) and returns
 * without synchronising.  A handle is not thread-safe: one handle per process x
 * device, as in the reference's one-process-per-GPU worker model
 * (call_modifications.py:405-414, 613-621).
 */
#ifndef DSP_B200_H
#define DSP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSP_B200_ABI_VERSION 1

typedef enum {
    DSP_OK = 0,
    DSP_ERR_INVALID = 1,     /* bad argument / unsupported shape */
    DSP_ERR_CUDA = 2,        /* a CUDA runtime or driver call failed */
    DSP_ERR_STATE = 3,       /* call order violated (e.g. forward before pack) */
    DSP_ERR_NOMEM = 4,
    DSP_ERR_UNSUPPORTED = 5  /* valid input this entry point does not cover; the caller has a general path */
} dsp_status;

/* module = ModelBiLSTM's `module` argument (models.py:120-128) */
typedef enum { DSP_BOTH_BILSTM = 0, DSP_SEQ_BILSTM = 1, DSP_SIGNAL_BILSTM = 2 } dsp_module;

/* Arithmetic of the recurrent/dense contractions.
 *   DSP_PRECISION_FP32: fp32 FMA on the CUDA cores (exact-order reference path).
 *   DSP_PRECISION_FP16: FP16 operands, fp32 accumulation in TMEM via tcgen05.mma,
 *                       fp32 cell state and gate math (the throughput path). */
typedef enum { DSP_PRECISION_FP32 = 0, DSP_PRECISION_FP16 = 1 } dsp_precision;

/* Mirrors the constructor arguments of ModelBiLSTM (models.py:103-106). */
typedef struct {
    int32_t seq_len;         /* 13 */
    int32_t signal_len;      /* 16 */
    int32_t num_layers1;     /* 3: layers of lstm_comb */
    int32_t num_layers2;     /* 1: layers of lstm_seq / lstm_signal */
    int32_t num_classes;     /* 2 */
    int32_t hidden_size;     /* 256 */
    int32_t vocab_size;      /* 16 */
    int32_t embedding_size;  /* 4 */
    int32_t is_base;         /* bool */
    int32_t is_signallen;    /* bool */
    int32_t module;          /* dsp_module */
    int32_t device;          /* CUDA ordinal */
    int32_t precision;       /* dsp_precision */
    int32_t reserved;
    int64_t max_batch;       /* sites per internal pass; workspace is sized for this */
} dsp_config;

typedef struct dsp_model_s* dsp_handle;

int dsp_abi_version(void);
const char* dsp_last_error(void);

/* ModelBiLSTM.__init__ (models.py:103-164): allocates the packed-weight arena and the
 * activation workspace for cfg->max_batch sites on cfg->device. */
int dsp_create(dsp_handle* out, const dsp_config* cfg);
int dsp_destroy(dsp_handle h);

/* load_state_dict (call_modifications.py:219-223): hand over one state_dict entry.
 * `name` is the reference's state_dict key (e.g. "lstm_comb.weight_hh_l1_reverse");
 * `host_data` is a HOST pointer to `numel` contiguous float32 values in torch's
 * row-major layout.  dsp_pack_weights() then converts everything that was set into the
 * kernel layouts (gate-interleaved, bias_ih+bias_hh pre-summed, FP16 tiles) and
 * uploads it; it fails with DSP_ERR_STATE if a key the configuration needs is missing. */
int dsp_set_param(dsp_handle h, const char* name, const float* host_data, int64_t numel);
int dsp_pack_weights(dsp_handle h);

/* ModelBiLSTM.forward (models.py:178-240) for n sites.
 *   kmer, base_means, base_stds, base_signal_lens: (n, seq_len) float32 (kmer holds
 *     float-coded base codes, cast like `kmer.long()`, models.py:186); may be NULL for
 *     signal_bilstm.   signals: (n, seq_len, signal_len) float32; may be NULL for seq_bilstm.
 *   states: NULL, or 6 device pointers {seq_h0, seq_c0, signal_h0, signal_c0, comb_h0,
 *     comb_c0}, each (num_layers*2, n, hidden) float32 indexed [layer*2+dir] -- the
 *     tensors init_hidden returns (models.py:169-176).  With NULL the initial states
 *     are drawn N(0,1) on the device from Philox4x32-10 keyed by (seed, site, slot),
 *     which is what the reference does statistically (fresh torch.randn per call).
 *   logits, probs: (n, num_classes) float32 outputs (forward returns both, :240).
 *   labels: optional (n) int32 = argmax of probs, first index on ties
 *     (torch.max(vlogits.data, 1), call_modifications.py:163); may be NULL. */
int dsp_forward(dsp_handle h,
                const float* kmer, const float* base_means, const float* base_stds,
                const float* base_signal_lens, const float* signals,
                const float* const* states, uint64_t seed, int64_t n,
                float* logits, float* probs, int32_t* labels, void* stream);

/* The same call with HOST buffers (the FloatTensor(...)/.cpu() boundary of _call_mods,
 * call_modifications.py:159-169): inputs are staged through pinned ring buffers and
 * copied host->device on a copy stream overlapped with compute, results are copied
 * back; returns after the outputs are valid on the host.  Initial states are always
 * Philox-drawn on the device. */
int dsp_forward_host(dsp_handle h,
                     const float* kmer, const float* base_means, const float* base_stds,
                     const float* base_signal_lens, const float* signals,
                     uint64_t seed, int64_t n,
                     float* logits, float* probs, int32_t* labels);

/* Asynchronous form for page-locked caller memory (every input and output buffer pinned):
 * submit enqueues the copies and kernels of one batch and returns a ticket at once; the
 * outputs are valid after dsp_forward_host_wait(h, ticket).  Submissions run in order and
 * overlap: batch i+1 crosses PCIe while batch i computes.  This is the streaming loop a
 * call_mods worker runs over successive feature batches (call_modifications.py:232-249). */
int dsp_forward_host_submit(dsp_handle h,
                            const float* kmer, const float* base_means, const float* base_stds,
                            const float* base_signal_lens, const float* signals,
                            uint64_t seed, int64_t n,
                            float* logits, float* probs, int32_t* labels, int64_t* ticket);
int dsp_forward_host_wait(dsp_handle h, int64_t ticket);

/* ---- training (train.py:104-128: model.train(), forward, loss.backward()) ------------------------
 * fp32 on the CUDA cores whatever cfg->precision says; the handle contributes its configuration only
 * (no dsp_set_param / dsp_pack_weights needed).  All pointers are DEVICE pointers; work is enqueued on
 * `stream`; nothing is allocated inside forward or backward.
 *
 * params: the module's parameters in state_dict order (models.py:131-161): embed.weight (unless
 *   signal_bilstm), lstm_seq.{weight_ih,weight_hh,bias_ih,bias_hh}_l{k}[_reverse] per layer, fc_seq.{weight,bias},
 *   the same for lstm_signal / fc_signal, lstm_comb, fc1, fc2 -- torch's row-major float32 layouts.
 *   dsp_train_shape gives their count and the number of dropout-mask slots.
 * dropout_masks: n_masks slots, each NULL (no dropout there) or a float32 tensor holding keep / (1 - p):
 *   slots [0, L2-1): lstm_seq inter-layer (n, seq_len, 2*nhid_seq) after layer l;  [L2-1, 2(L2-1)):
 *   lstm_signal likewise;  then L1-1 slots of lstm_comb (n, seq_len, 2*hidden);  then the head:
 *   (n, 2*hidden) before fc1 and (n, hidden) after fc1 (models.py:234-237).  L1 = num_layers1,
 *   L2 = num_layers2.  Backward must get the same masks as the forward whose arena it reads.
 * states: as for dsp_forward (6 pointers or NULL = Philox from `seed`); they are copied into the arena.
 *
 * Arena (saved activations of one forward, read by its backward; sections 256-byte aligned), per
 * LSTM stack of `layers` layers, hidden H, first-layer input K0:
 *   h0, c0: layers*2*n*H floats each; per layer l: y (n*T*2H), dropout output (n*T*2H, all but the last
 *   layer), gates i,f,g,o (n*T*8H), cell states (n*T*2H), the layer's weights in the forward kernel's
 *   layout 2 * ((ru(K,4) + ru(H,4))*4H + 4H) with K = K0 for l = 0, 2H otherwise;
 * then xseq (n*T*kseq) + kmer codes (n*T int32) when the module has the seq branch, signals (n*T*S)
 * when it has the signal branch, comb input (n*T*hidden), head: dropout(last states) (n*2*hidden),
 * fc1 output (n*hidden), relu(dropout(fc1)) (n*hidden).  dsp_train_arena_bytes returns the total:
 * for both_bilstm 13 x 16, hidden 256, 3 + 1 layers about 0.73 MB per site plus 19 MB of weights.
 * The workspace of dsp_train_backward is scratch only (dsp_train_workspace_bytes; ~0.3 MB per site for
 * the same model plus the split-K partial sums).
 *
 * dsp_train_forward writes logits (n, num_classes).  dsp_train_backward takes dlogits (n, num_classes),
 * the gradient of the loss w.r.t. the logits, and WRITES (does not add) every parameter's gradient to
 * grads[i] (same order and shapes as params; bias_ih and bias_hh receive the same values).  Sums over
 * sites use a fixed split and order: repeating a backward gives bit-identical gradients. */
int dsp_train_shape(dsp_handle h, int32_t* n_params, int32_t* n_masks);
int64_t dsp_train_arena_bytes(dsp_handle h, int64_t n);
int64_t dsp_train_workspace_bytes(dsp_handle h, int64_t n);
int dsp_train_forward(dsp_handle h, const float* const* params, int32_t n_params,
                      const float* kmer, const float* base_means, const float* base_stds,
                      const float* base_signal_lens, const float* signals,
                      const float* const* states, uint64_t seed, const float* const* dropout_masks,
                      int64_t n, void* arena, float* logits, void* stream);
int dsp_train_backward(dsp_handle h, const float* const* params, int32_t n_params,
                       const float* const* dropout_masks, const void* arena, const float* dlogits,
                       int64_t n, void* workspace, float* const* grads, void* stream);

/* Number of kernels this library launched on behalf of `h` since creation. */
int64_t dsp_launch_count(dsp_handle h);
/* Milliseconds (CUDA events on the launching stream) spent in kernels of class `which`
 * during the last dsp_forward when timing was enabled with dsp_set_timing(h, 1):
 * 0 = feature assembly/state init, 1 = recurrent layers (lstm_comb; all LSTM layers on the fp32 path),
 * 2 = per-timestep fc, 3 = head, 4 = branch recurrent layers (lstm_seq / lstm_signal, fp16 path).
 * Timing inserts event records only; it never synchronises inside dsp_forward. */
int dsp_set_timing(dsp_handle h, int enable);
int dsp_get_timing(dsp_handle h, int which, float* ms, int64_t* launches);

/* calculate_mods_frequency (call_mods_freq.py:29-74) for records already parsed into
 * columns (txt_formater.py:8-21).  All pointers are DEVICE pointers, n records in file
 * order:
 *   key   (uint64): site key = (chrom_id << 40) | pos, chrom_id assigned by the host;
 *   p0,p1 (double): the parsed probabilities;  label (int32): called_label.
 * Records with |p0-p1| < prob_cf are dropped (txt_formater.py:23-26).  Per key the
 * probabilities are summed in float64 strictly in record order (call_mods_freq.py:60-61);
 * counts are integers.  Outputs, one row per distinct key (capacity n), ordered by first
 * callable appearance (dict insertion order) when sort_by_key == 0 or by key value
 * when sort_by_key != 0:
 *   out_key, out_first (index of the first callable record of the key, which supplies
 *   strand / pos_in_strand / kmer, :55-59), out_p0, out_p1, out_met, out_unmet, out_cov.
 * *n_sites_host receives the number of rows (the call synchronises `stream`). */
int dsp_freq_aggregate(int device, const uint64_t* key, const double* p0, const double* p1,
                       const int32_t* label, int64_t n, double prob_cf, int sort_by_key,
                       uint64_t* out_key, int64_t* out_first, double* out_p0, double* out_p1,
                       int32_t* out_met, int32_t* out_unmet, int32_t* out_cov,
                       int64_t* n_sites_host, void* stream);

/* The same aggregation with HOST buffers, for a host that has no device-memory plumbing of its own (the call_freq
 * command line: no torch import in the process).  Inputs are the columns dsp_parse_calls writes: chrom_code (n) indexes
 * its name table; code_rank (n_codes, HOST) gives every code the rank of its name in the output's chromosome order
 * (Python string order for the reference's --sort, call_mods_freq.py:88) -- site key = (code_rank[chrom_code] << 40) | pos,
 * built on the device; pos must lie in [0, 2^40).  Outputs are HOST arrays of capacity out_cap (DSP_ERR_NOMEM with
 * *n_sites_host set if more sites than that).  Uploads, aggregation and download run on the default stream. */
int dsp_freq_aggregate_host(int device, const int32_t* chrom_code, const int64_t* code_rank, int32_t n_codes,
                            const int64_t* pos, const double* p0, const double* p1, const int32_t* label,
                            int64_t n, double prob_cf, int sort_by_key,
                            uint64_t* out_key, int64_t* out_first, double* out_p0, double* out_p1,
                            int32_t* out_met, int32_t* out_unmet, int32_t* out_cov, int64_t out_cap,
                            int64_t* n_sites_host);

/* Creates the CUDA context of `device` (a few hundred milliseconds in a fresh process).  The command lines call it from a
 * side thread while they parse their input, so that the first real call does not wait for it. */
int dsp_device_warmup(int device);

/* ---- multi-GPU call_freq: one process per GPU, records exchanged over NVLink peer memory -----------------
 * The reference's only parallel form of the aggregation is per-contig worker processes over temp files
 * (call_mods_freq.py:154-215, 262-295).  Here every rank parses a contiguous shard of the records (file order,
 * global record index = gidx_base + i) and the per-site reduction is sharded by site key: callable records go
 * to rank hash(key) % world, where they arrive grouped by source rank in file order and are summed in that
 * order -- the float64 sums are the reference's bit for bit, there is no partial-sum merge.
 *
 * A communicator owns two receive windows (window_bytes each) and a control block in device memory; the other
 * ranks of the box map them with CUDA IPC: export a blob on every rank, gather the blobs in rank order by any
 * means (torch.distributed.all_gather_object in the Python mirror), connect.  All ranks must then make the same
 * sequence of exchange calls (collective semantics).  A window that would overflow fails on every rank alike
 * with DSP_ERR_NOMEM and nothing is written; a peer that never arrives fails after 30 s with DSP_ERR_CUDA. */
typedef struct dsp_comm_s* dsp_comm;
int dsp_comm_create(dsp_comm* out, int device, int rank, int world, int64_t window_bytes);
int dsp_comm_export(dsp_comm c, void* blob, int64_t blob_cap, int64_t* blob_bytes);
int dsp_comm_connect(dsp_comm c, const void* blobs_in_rank_order, int64_t blob_bytes);
int dsp_comm_destroy(dsp_comm c);

/* calculate_mods_frequency (call_mods_freq.py:29-74) across the ranks of `c`.  DEVICE pointers: this rank's
 * n records in file order (columns as for dsp_freq_aggregate).  gidx_bounds_host (HOST, world + 1 ascending
 * values): rank r holds the global records [bounds[r], bounds[r+1]); gidx_base = bounds[rank].
 * Result: this rank's slice of the table as rows of 48 bytes
 *   { uint64 key; uint64 first (global index of the site's first callable record, which supplies strand /
 *     pos_in_strand / k-mer, :55-59); double prob_0 sum, prob_1 sum; int32 met, unmet, coverage, 0 }
 * in rows_out (DEVICE, capacity rows_cap), ordered by `first`: concatenating the ranks' slices in rank order gives
 * the reference's dict insertion order.  row_placement 0: the slices are ranges of `first` holding about the same
 * number of rows each, cut at splitters every rank derives from the same all-gathered sample (with reads in
 * random order nearly every site is first seen in rank 0's shard, so "send the row to the rank that parsed its
 * first record" would funnel the table through one GPU); row_placement 1: exactly that -- rank r receives the
 * rows whose `first` lies in its own shard [bounds[r], bounds[r+1]).  row_bounds_host (HOST, world + 1 values, may
 * be NULL) receives the ranges used.  *n_rows_host = rows written, *n_callable_host (may be NULL) = callable
 * records this rank RECEIVED.  Synchronises `stream`. */
int dsp_freq_aggregate_distributed(dsp_comm c, const uint64_t* key, const double* p0, const double* p1,
                                   const int32_t* label, int64_t n, uint64_t gidx_base, double prob_cf,
                                   const uint64_t* gidx_bounds_host, int32_t row_placement,
                                   void* rows_out, int64_t rows_cap, int64_t* n_rows_host,
                                   int64_t* n_callable_host, uint64_t* row_bounds_host, void* stream);

/* The exchange primitive on its own: n rows of row_bytes (48 or 96) in DEVICE memory; the row's uint64 at
 * field_offset selects the destination rank d with bounds[d] <= field < bounds[d+1] (bounds_host: world + 1
 * ascending values, HOST; bounds[0] and bounds[world] are not compared).  Rows keep their order per
 * (source, destination) and arrive concatenated in source-rank order in `out` (DEVICE, capacity out_cap_rows).
 * Used to bring finished site rows with their text columns to key-range owners for a --sort table
 * (call_mods_freq.py:87-90).  Synchronises `stream`. */
int dsp_comm_route_rows(dsp_comm c, const void* rows, int64_t n, int32_t row_bytes, int32_t field_offset,
                        const uint64_t* bounds_host, void* out, int64_t out_cap_rows, int64_t* n_out_host,
                        void* stream);

/* Milliseconds (CUDA events on the stream) of the last dsp_freq_aggregate_distributed call, 12 values: the four
 * stages (record exchange, local sort + replay, row exchange, ordering), then inside the record exchange and inside
 * the row exchange: count + scan + publish | waiting for every rank's counts | scatter over NVLink | signal +
 * waiting for every rank's stores. */
int dsp_comm_last_timing(dsp_comm c, float* ms12);

/* dsp_parse_calls: ModRecord.__init__ (utils/txt_formater.py:8-21) for a whole call_mods file held in memory
 * (HOST pointers): every line is strip()-ed and split on tabs; columns 1, 3, 8 are parsed like int(), 6 and 7
 * like float() (correctly rounded to float64), chromosome names (column 0) are interned -- chrom_code[i] indexes
 * the '\n'-separated list written to `names` (*n_names entries, *names_bytes bytes; DSP_ERR_NOMEM if names_cap
 * is too small) -- strand (column 2) and k_mer (column 9) are copied into zero-padded cells of 4 and 24 bytes
 * (a longer value returns DSP_ERR_UNSUPPORTED).  Columns beyond the tenth are ignored; fewer than ten, an empty
 * line inside the file or an unparsable number return DSP_ERR_INVALID (the reference raises).  With
 * max_records == 0 only the lines are counted (*n_records) and no output pointer is touched. */
int dsp_parse_calls(const char* text, int64_t nbytes, int64_t max_records,
                    int32_t* chrom_code, int64_t* pos, char* strand, int64_t* pos_in_strand,
                    double* p0, double* p1, int32_t* label, char* kmer,
                    char* names, int64_t names_cap, int64_t* names_bytes, int32_t* n_names,
                    int64_t* n_records, int32_t nthreads);

/* dsp_format_freq: the text of write_sitekey2stats (call_mods_freq.py:87-120) for n sites already in output order
 * (HOST pointers).  chrom_text / strand_text / kmer_text hold the n strings of the column joined by '\n',
 * NUL-terminated.  Sites with coverage 0 are skipped (:104).  is_bed == 0: the 11-column table
 * "%s\t%d\t%s\t%d\t%.3f\t%.3f\t%d\t%d\t%d\t%.4f\t%s" (:112-118); else the bedMethyl line of :106-110
 * with percent = int(round(met / coverage * 100 + 0.001, 0)).  *out_bytes receives the size needed;
 * DSP_ERR_NOMEM if out_cap is too small. */
int dsp_format_freq(const char* chrom_text, const char* strand_text, const char* kmer_text,
                    const int64_t* pos, const int64_t* pos_in_strand, const double* prob_0, const double* prob_1,
                    const int32_t* met, const int32_t* unmet, const int32_t* coverage, int64_t n, int32_t is_bed,
                    char* out, int64_t out_cap, int64_t* out_bytes, int32_t nthreads);

/* dsp_freq_aggregate keeps its scratch device memory cached between calls; this frees it. */
int dsp_freq_release_cache(void);

/* ---- text boundary of call_mods (host code, HOST pointers) ---------------------------------
 * dsp_parse_features: _read_features_file (call_modifications.py:55-127) for a block of the
 * feature file written by `deepsignal_plant extract` (12 tab-separated columns,
 * extract_features.py:381-395), parsed straight into caller buffers (typically page-locked,
 * then handed to dsp_forward_host_submit).  Only complete lines are consumed unless
 * is_final != 0; at most max_sites lines.  The first six columns of line i -- the "sampleinfo"
 * its output line starts with (:89) -- are packed into info_text at
 * [info_off[i], info_off[i+1]) (info_off has max_sites + 1 entries; DSP_ERR_NOMEM if info_cap
 * is too small).  Numbers follow Python: float(x) to double, then float32; k-mer letters go
 * through base2code_dna (utils/process_utils.py:22-29).  Malformed lines fail with
 * DSP_ERR_INVALID (the reference raises).  *consumed = bytes of `text` used. */
int dsp_parse_features(const char* text, int64_t nbytes, int32_t is_final,
                       int32_t seq_len, int32_t signal_len, int64_t max_sites,
                       float* kmer, float* base_means, float* base_stds, float* base_signal_lens,
                       float* signals, int32_t* labels,
                       char* info_text, int64_t info_cap, int64_t* info_off,
                       int64_t* n_sites, int64_t* consumed, int32_t nthreads);

/* dsp_format_calls: the per-site output loop of _call_mods (call_modifications.py:175-188):
 *   sampleinfo \t prob_0 \t prob_1 \t label \t 5-mer \n
 * with prob_0 = round(p0/(p0+p1), 6), prob_1 = round(1 - prob_0, 6) evaluated in float32 and
 * printed like str(numpy.float32); the 5-mer is kmer[c-2:c+3] of the (n, seq_len) float-coded
 * k-mer array.  probs is (n, 2) float32, labels (n) int32; info_text / info_off come from
 * dsp_parse_features.  *out_bytes receives the size needed; DSP_ERR_NOMEM if out_cap is too
 * small. */
int dsp_format_calls(const char* info_text, const int64_t* info_off, const float* kmer,
                     int32_t seq_len, const float* probs, const int32_t* labels, int64_t n,
                     char* out, int64_t out_cap, int64_t* out_bytes, int32_t nthreads);

/* The sample-info columns of sites extracted by dsp_extract_features, i.e. what
 * _read_features_from_fast5s joins per site (call_modifications.py:312):
 *   chrom \t pos \t alignstrand \t pos_in_strand \t readname \t strand
 * packed into info_text / info_off exactly as dsp_parse_features leaves them (n + 1 offsets), ready
 * for dsp_format_calls.  HOST pointers.  Per read r: chrom = chrom_text[chrom_off[r] .. chrom_off[r+1]),
 * readname likewise, alignstrand[r] and strand[r] one character each ('+'/'-', 't'/'c'); per site:
 * site_read, pos, pos_in_strand.  DSP_ERR_NOMEM if info_cap is too small. */
int dsp_format_sampleinfo(const char* chrom_text, const int64_t* chrom_off, const char* name_text, const int64_t* name_off,
                          const char* alignstrand, const char* strand,
                          const int32_t* site_read, const int64_t* pos, const int64_t* pos_in_strand, int64_t n,
                          char* info_text, int64_t info_cap, int64_t* info_off, int32_t nthreads);

/* ---- feature extraction from decoded re-squiggled reads (SURVEY.md 8(f) row 4) ----------------
 * dsp_extract_features: the numeric body of _extract_features (extract_features.py:280-378) for a
 * batch of reads whose fast5 content is already decoded into flat DEVICE arrays:
 *   raw (int16 DAC samples of all reads, concatenated), raw_off (n_reads + 1 offsets into raw),
 *   scaling / offset (per read, float64: _get_scaling_of_a_read, :255-273; a NaN scaling = no channel
 *   info, samples used as they are, :313-315);
 *   the tombo event tables of all reads, concatenated: ev_start (relative to the read's first raw
 *   sample, read_start_rel_to_raw already added as :80 does), ev_len, ev_base (ASCII letters);
 *   the sites to extract: site_read (read index) and site_ev (index of the site's own event in the
 *   concatenated table; the seq_len events centred on it must belong to the same read, which is the
 *   `num_bases <= loc < len - num_bases` rule of :341).
 * Per read: _rescale_signals (:276-277) and _normalize_signals (:179-190) with normalize_method 0 =
 * 'mad' (median / statsmodels.robust.mad) or 1 = 'zscore' (np.mean / np.std), float64, then
 * np.around(., 6); their shift and scale are left in read_shift / read_scale (n_reads doubles each).  Per site and base: len, np.mean, np.std
 * (float64, numpy's pairwise summation order) and the seq_len x signal_len rectangle of
 * _get_signals_rect (:232-251), written as float32 into the five tensors dsp_forward takes
 * (kmer = base2code_dna codes).  round_stats != 0 rounds means/stds to 6 decimals first, which is
 * what the feature FILE carries (_features_to_str, :388-389); 0 is the direct fast5 route
 * (call_modifications.py:309-318).  Bases with more than signal_len samples are subsampled in order:
 * with `drawn` (n_sites x seq_len x signal_len int32 offsets, rows of other bases ignored) the given
 * offsets are used -- the way to replay the reference's random.sample draws; with NULL an ordered
 * uniform subset is drawn on the device from Philox4x32-10 keyed by (seed, site, base), which is what
 * the reference does statistically.  Enqueues on `stream`; does not synchronise. */
int dsp_extract_features(int device,
                         const int16_t* raw, const int64_t* raw_off, const double* scaling, const double* offset,
                         int64_t n_reads,
                         const int64_t* ev_start, const int64_t* ev_len, const uint8_t* ev_base,
                         const int32_t* site_read, const int64_t* site_ev, int64_t n_sites,
                         int32_t seq_len, int32_t signal_len, int32_t normalize_method, int32_t round_stats,
                         const int32_t* drawn, uint64_t seed,
                         double* read_shift, double* read_scale,
                         float* kmer, float* base_means, float* base_stds, float* base_signal_lens,
                         float* signals, void* stream);

/* dsp_extract_features_f64: the same call with float64 outputs -- the values the reference holds before
 * FloatTensor narrows them, needed where they are PRINTED (the feature file of `deepsignal_plant extract`):
 * all five outputs are double (kmer codes and lens included). */
int dsp_extract_features_f64(int device,
                             const int16_t* raw, const int64_t* raw_off, const double* scaling, const double* offset,
                             int64_t n_reads,
                             const int64_t* ev_start, const int64_t* ev_len, const uint8_t* ev_base,
                             const int32_t* site_read, const int64_t* site_ev, int64_t n_sites,
                             int32_t seq_len, int32_t signal_len, int32_t normalize_method, int32_t round_stats,
                             const int32_t* drawn, uint64_t seed,
                             double* read_shift, double* read_scale,
                             double* kmer, double* base_means, double* base_stds, double* base_signal_lens,
                             double* signals, void* stream);

/* dsp_format_features: _features_to_str (extract_features.py:381-395) for n sites, HOST pointers:
 *   sampleinfo \t k_mer \t means \t stds \t lens \t signals \t methy_label \n
 * info_text / info_off as dsp_format_sampleinfo writes them; kmer_letters (n, seq_len) ASCII; means, stds,
 * lens (n, seq_len) and signals (n, seq_len, signal_len) as dsp_extract_features_f64 produced them with
 * round_stats = 1.  Numbers are printed like str(numpy.float64) (shortest round-trip digits, positional in
 * [1e-4, 1e16), scientific otherwise), lens as integers.  *out_bytes receives the size needed;
 * DSP_ERR_NOMEM if out_cap is too small. */
int dsp_format_features(const char* info_text, const int64_t* info_off, const uint8_t* kmer_letters,
                        const double* means, const double* stds, const double* lens, const double* signals,
                        int32_t methy_label, int64_t n, int32_t seq_len, int32_t signal_len,
                        char* out, int64_t out_cap, int64_t* out_bytes, int32_t nthreads);

/* dsp_find_sites: which bases of a batch of decoded reads are targets --
 * get_refloc_of_methysite_in_motif (utils/process_utils.py:97-112) over every read, then the site filters
 * of _extract_features in its order (extract_features.py:341-352): a margin of (seq_len-1)/2 bases at both
 * read ends, the strand-aware genome position, the optional region.  DEVICE pointers except `motifs`
 * (HOST: n_motifs x motif_len ASCII letters, the expanded list get_motif_seqs returns) and n_sites_host.
 *   ev_base / ev_off: the concatenated event tables as in dsp_extract_features (n_events letters);
 *   per read: chrom_start (mapped_start), minus_strand (1 when mapped_strand is '-'), chrom_len (contig
 *   length, < 0 or NULL pointer = unknown -> pos_in_strand -1), and, when a region is given, the half-open
 *   position range [region_start, region_end) the read may contribute (an empty range for reads on other
 *   contigs; both NULL = no region).
 * Outputs (capacity max_sites), in the reference's order (reads in order, positions ascending in the read):
 *   site_read, site_ev (what dsp_extract_features takes), pos, pos_in_strand.  *n_sites_host receives the
 *   number found (the call synchronises `stream`); DSP_ERR_NOMEM, with nothing written, if it exceeds max_sites.
 * The --positions set filter of :354 is a host-side string-set lookup and stays with the caller. */
int dsp_find_sites(int device, const uint8_t* ev_base, const int64_t* ev_off, int64_t n_reads, int64_t n_events,
                   const char* motifs, int32_t n_motifs, int32_t motif_len, int32_t methyloc, int32_t seq_len,
                   const int64_t* chrom_start, const uint8_t* minus_strand, const int64_t* chrom_len,
                   const int64_t* region_start, const int64_t* region_end, int64_t max_sites,
                   int32_t* site_read, int64_t* site_ev, int64_t* pos, int64_t* pos_in_strand,
                   int64_t* n_sites_host, void* stream);

/* Known-answer test of the tcgen05/TMEM/bulk-copy building blocks on `device`: a one-CTA
 * FP16 GEMM with FP32 accumulation checked against a double-precision host product.
 * which: 0,1 = both operands from shared memory; 2,3 = A operand staged in TMEM.
 * *max_abs_err receives the largest absolute deviation. */
int dsp_selftest(int device, int which, double* max_abs_err);

#ifdef __cplusplus
}
#endif
#endif /* DSP_B200_H */
