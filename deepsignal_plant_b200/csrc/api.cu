// C ABI of libdsp_b200 (include/dsp_b200.h): handle life cycle, weight packing,
// forward orchestration, host-buffer streaming.  The arithmetic lives in kernels_f32.cu
// (CUDA-core fp32) and kernels_tc.cu (tcgen05 FP16 operands).
#include "common.cuh"
#include "tc.cuh"
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <new>

namespace dsp {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

namespace {

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int dev_alloc(Model* m, void** p, size_t bytes) {
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) {
        set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
        return DSP_ERR_NOMEM;
    }
    m->device_allocs.push_back(*p);
    return DSP_OK;
}

int upload(Model* m, float** dst, const std::vector<float>& host) {
    int rc = dev_alloc(m, (void**)dst, host.size() * sizeof(float));
    if (rc) return rc;
    DSP_CUDA(cudaMemcpy(*dst, host.data(), host.size() * sizeof(float), cudaMemcpyHostToDevice));
    return DSP_OK;
}

const std::vector<float>* find_param(Model* m, const std::string& name, int64_t numel) {
    auto it = m->params.find(name);
    if (it == m->params.end()) {
        set_error("state_dict entry '%s' was not set before dsp_pack_weights", name.c_str());
        return nullptr;
    }
    if ((int64_t)it->second.size() != numel) {
        set_error("state_dict entry '%s' has %zu elements, expected %lld", name.c_str(), it->second.size(),
                  (long long)numel);
        return nullptr;
    }
    return &it->second;
}

// nn.LSTM parameters of one stack -> kernel layouts.
int pack_lstm_stack(Model* m, const char* prefix, int num_layers, int in0, int H,
                    std::vector<LstmLayer>& out) {
    out.clear();
    for (int l = 0; l < num_layers; ++l) {
        LstmLayer L;
        L.K = (l == 0) ? in0 : 2 * H;
        L.H = H;
        const int Kp = ru(L.K, 4), Hp = ru(H, 4);
        const std::vector<float>* raw[2][4];
        for (int d = 0; d < 2; ++d) {
            char name[128];
            const char* sfx = d ? "_reverse" : "";
            snprintf(name, sizeof(name), "%s.weight_ih_l%d%s", prefix, l, sfx);
            const std::vector<float>* wih = find_param(m, name, (int64_t)4 * H * L.K);
            snprintf(name, sizeof(name), "%s.weight_hh_l%d%s", prefix, l, sfx);
            const std::vector<float>* whh = find_param(m, name, (int64_t)4 * H * H);
            snprintf(name, sizeof(name), "%s.bias_ih_l%d%s", prefix, l, sfx);
            const std::vector<float>* bih = find_param(m, name, (int64_t)4 * H);
            snprintf(name, sizeof(name), "%s.bias_hh_l%d%s", prefix, l, sfx);
            const std::vector<float>* bhh = find_param(m, name, (int64_t)4 * H);
            if (!wih || !whh || !bih || !bhh) return DSP_ERR_STATE;
            raw[d][0] = wih; raw[d][1] = whh; raw[d][2] = bih; raw[d][3] = bhh;
            std::vector<float> wt((size_t)(Kp + Hp) * 4 * H, 0.f), bias((size_t)4 * H);
            for (int g = 0; g < 4; ++g)
                for (int j = 0; j < H; ++j) {
                    const int row = g * H + j;
                    for (int k = 0; k < L.K; ++k) wt[((size_t)k * 4 + g) * H + j] = (*wih)[(size_t)row * L.K + k];
                    for (int k = 0; k < H; ++k) wt[((size_t)(Kp + k) * 4 + g) * H + j] = (*whh)[(size_t)row * H + k];
                    bias[row] = (*bih)[row] + (*bhh)[row];
                }
            int rc = upload(m, &L.f32[d].wt, wt);
            if (rc) return rc;
            rc = upload(m, &L.f32[d].bias, bias);
            if (rc) return rc;
        }
        if (m->cfg.precision == DSP_PRECISION_FP16) {
            // lstm_seq layer 0: columns [E, E + 2|3) are mean, std(, len) (models.py:188-195)
            const bool split = l == 0 && strcmp(prefix, "lstm_seq") == 0 && tc_seq_split(m);
            const int e = m->cfg.is_base ? m->cfg.embedding_size : 0, nsc = m->cfg.is_signallen ? 3 : 2;
            int rc = tc_pack_lstm_layer(m, L, raw[0][0]->data(), raw[0][1]->data(), raw[0][2]->data(), raw[0][3]->data(),
                                        raw[1][0]->data(), raw[1][1]->data(), raw[1][2]->data(), raw[1][3]->data(),
                                        split ? e : 0, split ? nsc : 0, (split && m->cfg.is_signallen) ? e + 2 : -1);
            if (rc) return rc;
        }
        out.push_back(L);
    }
    return DSP_OK;
}

// kind: 0 = fp32 layout only, 1 = also a tensor-core per-timestep fc, 2 = also the tensor-core head (fc1)
int pack_dense(Model* m, const char* prefix, int K, int J, DenseF32& D, int kind) {
    std::string wn = std::string(prefix) + ".weight", bn = std::string(prefix) + ".bias";
    const std::vector<float>* w = find_param(m, wn, (int64_t)J * K);
    const std::vector<float>* b = find_param(m, bn, J);
    if (!w || !b) return DSP_ERR_STATE;
    D.K = K; D.J = J;
    const int Kp = ru(K, 4);
    std::vector<float> wt((size_t)Kp * J, 0.f);
    for (int j = 0; j < J; ++j)
        for (int k = 0; k < K; ++k) wt[(size_t)k * J + j] = (*w)[(size_t)j * K + k];
    int rc = upload(m, &D.wt, wt);
    if (rc) return rc;
    rc = upload(m, &D.bias, *b);
    if (rc) return rc;
    if (m->cfg.precision == DSP_PRECISION_FP16 && kind != 0) {
        rc = (kind == 2) ? tc_pack_head(m, D, w->data(), b->data()) : tc_pack_dense(m, D, w->data(), b->data());
        if (rc) return rc;
    }
    return DSP_OK;
}

bool has_seq(const Model* m) { return m->cfg.module != DSP_SIGNAL_BILSTM; }
bool has_signal(const Model* m) { return m->cfg.module != DSP_SEQ_BILSTM; }

struct StateGroup { int layers; int hidden; };

void state_groups(const Model* m, StateGroup g[3]) {
    g[0] = {has_seq(m) ? m->cfg.num_layers2 : 0, m->nhid_seq};
    g[1] = {has_signal(m) ? m->cfg.num_layers2 : 0, m->nhid_signal};
    g[2] = {m->cfg.num_layers1, m->cfg.hidden_size};
}

// One pass over n <= cap sites whose inputs already sit on the device.
// states6: per group h0/c0 base pointers for THIS chunk and the dir stride (floats) of
// each group; nullptr -> Philox.
int forward_chunk(Model* m, const float* kmer, const float* means, const float* stds, const float* lens,
                  const float* signals, const float* const* states6, const int64_t* state_stride,
                  uint64_t seed, uint64_t chunk_id, int64_t n, float* logits, float* probs, int32_t* labels,
                  cudaStream_t st) {
    const dsp_config& c = m->cfg;
    const int T = c.seq_len, H = c.hidden_size;
    StateGroup grp[3];
    state_groups(m, grp);
    const float* h0[3]; const float* c0[3]; int64_t sstride[3];
    if (!states6 && c.precision == DSP_PRECISION_FP16)      // states are drawn inside the layer kernels
        return tc_forward_chunk(m, kmer, means, stds, lens, signals, nullptr, nullptr, nullptr, seed, chunk_id, n,
                                logits, probs, labels, st);
    if (states6) {
        for (int g = 0; g < 3; ++g) { h0[g] = states6[2 * g]; c0[g] = states6[2 * g + 1]; sstride[g] = state_stride[g]; }
    } else {
        Span sp(m, 0, st);
        float* p = m->states;
        int64_t total = 0;
        for (int g = 0; g < 3; ++g) {
            int64_t cnt = (int64_t)grp[g].layers * 2 * n * grp[g].hidden;
            h0[g] = p + total; total += cnt;
            c0[g] = p + total; total += cnt;
            sstride[g] = n * grp[g].hidden;
        }
        int rc = philox_normal(m, m->states, total, seed, chunk_id, st);
        if (rc) return rc;
    }
    if (c.precision == DSP_PRECISION_FP16)
        return tc_forward_chunk(m, kmer, means, stds, lens, signals, h0, c0, sstride, seed, chunk_id, n, logits, probs, labels, st);

    int rc;
    int comb_off = 0;
    if (has_seq(m)) {
        { Span sp(m, 0, st); rc = f32_assemble_seq(m, kmer, means, stds, lens, n, m->xseq, st); if (rc) return rc; }
        const float* x = m->xseq; int xs = T * m->kseq, xt = m->kseq;
        int hs = m->nhid_seq;
        for (int l = 0; l < c.num_layers2; ++l) {
            Span sp(m, 1, st);
            rc = f32_lstm_layer(m, m->lstm_seq[l], x, xs, xt, h0[0] + (int64_t)l * 2 * sstride[0],
                                c0[0] + (int64_t)l * 2 * sstride[0], sstride[0], m->buf[l & 1], n, st);
            if (rc) return rc;
            x = m->buf[l & 1]; xs = T * 2 * hs; xt = 2 * hs;
        }
        { Span sp(m, 2, st); rc = f32_dense(m, m->fc_seq, x, n * T, 2 * hs, m->comb_in, H, 1, st); if (rc) return rc; }
        comb_off = hs;
    }
    if (has_signal(m)) {
        const float* x = signals; int xs = T * c.signal_len, xt = c.signal_len;
        int hs = m->nhid_signal;
        for (int l = 0; l < c.num_layers2; ++l) {
            Span sp(m, 1, st);
            rc = f32_lstm_layer(m, m->lstm_signal[l], x, xs, xt, h0[1] + (int64_t)l * 2 * sstride[1],
                                c0[1] + (int64_t)l * 2 * sstride[1], sstride[1], m->buf[l & 1], n, st);
            if (rc) return rc;
            x = m->buf[l & 1]; xs = T * 2 * hs; xt = 2 * hs;
        }
        { Span sp(m, 2, st); rc = f32_dense(m, m->fc_signal, x, n * T, 2 * hs, m->comb_in + comb_off, H, 1, st); if (rc) return rc; }
    }
    const float* x = m->comb_in; int xs = T * H, xt = H;
    for (int l = 0; l < c.num_layers1; ++l) {
        Span sp(m, 1, st);
        rc = f32_lstm_layer(m, m->lstm_comb[l], x, xs, xt, h0[2] + (int64_t)l * 2 * sstride[2],
                            c0[2] + (int64_t)l * 2 * sstride[2], sstride[2], m->buf[l & 1], n, st);
        if (rc) return rc;
        x = m->buf[l & 1]; xs = T * 2 * H; xt = 2 * H;
    }
    { Span sp(m, 3, st); rc = f32_head(m, x, n, logits, probs, labels, st); if (rc) return rc; }
    return DSP_OK;
}

bool is_device_accessible_host(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

}  // namespace
}  // namespace dsp

using namespace dsp;

extern "C" {

int dsp_abi_version(void) { return DSP_B200_ABI_VERSION; }
const char* dsp_last_error(void) { return g_err; }

int dsp_create(dsp_handle* out, const dsp_config* cfg) {
    DSP_REQUIRE(out && cfg, DSP_ERR_INVALID, "dsp_create: null argument");
    *out = nullptr;
    DSP_REQUIRE(cfg->seq_len >= 1 && cfg->signal_len >= 1 && cfg->num_layers1 >= 1 && cfg->num_layers2 >= 1 &&
                cfg->num_classes >= 1 && cfg->hidden_size >= 2 && cfg->vocab_size >= 1 && cfg->embedding_size >= 1,
                DSP_ERR_INVALID, "dsp_create: non-positive dimension in config");
    DSP_REQUIRE(cfg->module >= DSP_BOTH_BILSTM && cfg->module <= DSP_SIGNAL_BILSTM, DSP_ERR_INVALID,
                "--model_type is not right!");
    DSP_REQUIRE(cfg->precision == DSP_PRECISION_FP32 || cfg->precision == DSP_PRECISION_FP16, DSP_ERR_INVALID,
                "dsp_create: unknown precision %d", cfg->precision);
    DSP_REQUIRE(cfg->max_batch >= 1, DSP_ERR_INVALID, "dsp_create: max_batch must be >= 1");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        set_error("dsp_create: no CUDA device available (%s); this library has no CPU path",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        cudaGetLastError();
        return DSP_ERR_CUDA;
    }
    DSP_REQUIRE(cfg->device >= 0 && cfg->device < ndev, DSP_ERR_INVALID, "dsp_create: device %d out of range (%d)",
                cfg->device, ndev);
    DeviceGuard guard(cfg->device);
    cudaDeviceProp prop;
    DSP_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
    DSP_REQUIRE(prop.major == 10, DSP_ERR_INVALID,
                "dsp_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", cfg->device,
                prop.major, prop.minor);
    dsp_model_s* m = new (std::nothrow) dsp_model_s();
    DSP_REQUIRE(m, DSP_ERR_NOMEM, "dsp_create: out of host memory");
    m->cfg = *cfg;
    const int H = cfg->hidden_size;
    if (cfg->module == DSP_BOTH_BILSTM) { m->nhid_seq = H / 2; m->nhid_signal = H - H / 2; }
    else if (cfg->module == DSP_SEQ_BILSTM) { m->nhid_seq = H; }
    else { m->nhid_signal = H; }
    m->kseq = (cfg->is_base ? cfg->embedding_size : 0) + (cfg->is_signallen ? 3 : 2);
    m->cap = cfg->max_batch;
    m->n_sm = prop.multiProcessorCount;
    const int T = cfg->seq_len;
    int rc = DSP_OK;
    StateGroup grp[3];
    state_groups(m, grp);
    for (int g = 0; g < 3; ++g) m->state_floats_per_site += (int64_t)grp[g].layers * 2 * grp[g].hidden * 2;
    do {
        if ((rc = dev_alloc(m, (void**)&m->states, sizeof(float) * m->cap * m->state_floats_per_site))) break;
        if (cfg->precision == DSP_PRECISION_FP32) {
            if ((rc = dev_alloc(m, (void**)&m->xseq, sizeof(float) * m->cap * T * m->kseq))) break;
            if ((rc = dev_alloc(m, (void**)&m->buf[0], sizeof(float) * m->cap * T * 2 * H))) break;
            if ((rc = dev_alloc(m, (void**)&m->buf[1], sizeof(float) * m->cap * T * 2 * H))) break;
            if ((rc = dev_alloc(m, (void**)&m->comb_in, sizeof(float) * m->cap * T * H))) break;
        } else {
            if ((rc = tc_create(m))) break;
        }
    } while (0);
    if (rc) { dsp_destroy(m); return rc; }
    m->n_workspace_allocs = m->device_allocs.size();
    *out = m;
    return DSP_OK;
}

int dsp_destroy(dsp_handle h) {
    if (!h) return DSP_OK;
    dsp_model_s* m = h;
    DeviceGuard guard(m->cfg.device);
    cudaDeviceSynchronize();
    tc_destroy(m);
    for (void* p : m->device_allocs) cudaFree(p);
    for (int i = 0; i < Model::NBUF; ++i) {
        if (m->pinned_in[i]) cudaFreeHost(m->pinned_in[i]);
        if (m->pinned_out[i]) cudaFreeHost(m->pinned_out[i]);
        if (m->dev_in[i]) cudaFree(m->dev_in[i]);
        if (m->dev_out[i]) cudaFree(m->dev_out[i]);
        if (m->ev_h2d[i]) cudaEventDestroy(m->ev_h2d[i]);
        if (m->ev_done[i]) cudaEventDestroy(m->ev_done[i]);
    }
    for (int i = 0; i < Model::NTICKET; ++i) if (m->ev_ticket[i]) cudaEventDestroy(m->ev_ticket[i]);
    for (int i = 0; i < Model::NBUF; ++i) if (m->ev_computed[i]) cudaEventDestroy(m->ev_computed[i]);
    if (m->copy_stream) cudaStreamDestroy(m->copy_stream);
    if (m->compute_stream) cudaStreamDestroy(m->compute_stream);
    if (m->d2h_stream) cudaStreamDestroy(m->d2h_stream);
    for (cudaEvent_t e : m->event_pool) cudaEventDestroy(e);
    cudaGetLastError();
    delete m;
    return DSP_OK;
}

int dsp_set_param(dsp_handle h, const char* name, const float* host_data, int64_t numel) {
    DSP_REQUIRE(h && name && host_data && numel >= 0, DSP_ERR_INVALID, "dsp_set_param: null argument");
    h->params[name].assign(host_data, host_data + numel);
    h->packed = false;
    return DSP_OK;
}

int dsp_pack_weights(dsp_handle h) {
    DSP_REQUIRE(h, DSP_ERR_INVALID, "dsp_pack_weights: null handle");
    Model* m = h;
    DeviceGuard guard(m->cfg.device);
    const dsp_config& c = m->cfg;
    // re-packing after another load_state_dict: free the previous weight arena (the workspace stays)
    if (m->device_allocs.size() > m->n_workspace_allocs) {
        DSP_CUDA(cudaDeviceSynchronize());
        for (size_t i = m->n_workspace_allocs; i < m->device_allocs.size(); ++i) cudaFree(m->device_allocs[i]);
        m->device_allocs.resize(m->n_workspace_allocs);
        tc_drop_packs(m);
        m->embed = nullptr;
        m->packed = false;
    }
    int rc;
    const int H = c.hidden_size;
    if (has_seq(m)) {
        if (c.is_base) {
            const std::vector<float>* e = find_param(m, "embed.weight", (int64_t)c.vocab_size * c.embedding_size);
            if (!e) return DSP_ERR_STATE;
            if ((rc = upload(m, &m->embed, *e))) return rc;
        }
        if ((rc = pack_lstm_stack(m, "lstm_seq", c.num_layers2, m->kseq, m->nhid_seq, m->lstm_seq))) return rc;
        if ((rc = pack_dense(m, "fc_seq", 2 * m->nhid_seq, m->nhid_seq, m->fc_seq, 1))) return rc;
    }
    if (has_signal(m)) {
        if ((rc = pack_lstm_stack(m, "lstm_signal", c.num_layers2, c.signal_len, m->nhid_signal, m->lstm_signal))) return rc;
        if ((rc = pack_dense(m, "fc_signal", 2 * m->nhid_signal, m->nhid_signal, m->fc_signal, 1))) return rc;
    }
    if ((rc = pack_lstm_stack(m, "lstm_comb", c.num_layers1, H, H, m->lstm_comb))) return rc;
    if ((rc = pack_dense(m, "fc1", 2 * H, H, m->fc1, 2))) return rc;
    if ((rc = pack_dense(m, "fc2", H, c.num_classes, m->fc2, 0))) return rc;
    DSP_CUDA(cudaDeviceSynchronize());
    m->packed = true;
    return DSP_OK;
}

int dsp_forward(dsp_handle h, const float* kmer, const float* base_means, const float* base_stds,
                const float* base_signal_lens, const float* signals, const float* const* states,
                uint64_t seed, int64_t n, float* logits, float* probs, int32_t* labels, void* stream) {
    DSP_REQUIRE(h, DSP_ERR_INVALID, "dsp_forward: null handle");
    Model* m = h;
    DSP_REQUIRE(m->packed, DSP_ERR_STATE, "dsp_forward: weights not packed (call dsp_pack_weights after dsp_set_param)");
    DSP_REQUIRE(n >= 0, DSP_ERR_INVALID, "dsp_forward: negative batch");
    if (n == 0) return DSP_OK;
    DSP_REQUIRE(logits && probs, DSP_ERR_INVALID, "dsp_forward: null output pointer");
    if (has_seq(m)) DSP_REQUIRE(kmer && base_means && base_stds && base_signal_lens, DSP_ERR_INVALID,
                                "dsp_forward: sequence features are required for this module");
    if (has_signal(m)) DSP_REQUIRE(signals, DSP_ERR_INVALID, "dsp_forward: signals are required for this module");
    DeviceGuard guard(m->cfg.device);
    cudaStream_t st = (cudaStream_t)stream;
    const dsp_config& c = m->cfg;
    const int T = c.seq_len, C = c.num_classes;
    if (m->timing) { m->spans.clear(); m->event_next = 0; }
    StateGroup grp[3];
    state_groups(m, grp);
    uint64_t chunk_id = 0;
    for (int64_t s = 0; s < n; s += m->cap, ++chunk_id) {
        const int64_t cn = (n - s < m->cap) ? (n - s) : m->cap;
        const float* st6[6]; int64_t stride[3];
        if (states) {
            for (int g = 0; g < 3; ++g) {
                stride[g] = n * grp[g].hidden;
                if (grp[g].layers > 0) {
                    DSP_REQUIRE(states[2 * g] && states[2 * g + 1], DSP_ERR_INVALID, "dsp_forward: states[%d] is null", 2 * g);
                    st6[2 * g] = states[2 * g] + s * grp[g].hidden;
                    st6[2 * g + 1] = states[2 * g + 1] + s * grp[g].hidden;
                } else { st6[2 * g] = st6[2 * g + 1] = nullptr; }
            }
        }
        int rc = forward_chunk(m, kmer ? kmer + s * T : nullptr, base_means ? base_means + s * T : nullptr,
                               base_stds ? base_stds + s * T : nullptr,
                               base_signal_lens ? base_signal_lens + s * T : nullptr,
                               signals ? signals + s * T * c.signal_len : nullptr,
                               states ? st6 : nullptr, stride, seed, chunk_id, cn,
                               logits + s * C, probs + s * C, labels ? labels + s : nullptr, st);
        if (rc) return rc;
    }
    return DSP_OK;
}

// Host-buffer path.  The batch is cut into chunks of host_chunk sites (two full waves of CTA
// pairs); chunk i+1 crosses PCIe on the copy stream while chunk i computes, through a ring of
// NBUF device buffers that is carried across calls, so that back-to-back submissions overlap too.
// Pinned (device-accessible) caller memory is copied from / to directly; pageable memory is staged
// through pinned buffers of the library (synchronous entry point only).
static int host_setup(Model* m) {
    if (m->copy_stream) return DSP_OK;
    const dsp_config& c = m->cfg;
    const int T = c.seq_len, S = c.signal_len, C = c.num_classes;
    const int64_t two_waves = (int64_t)m->n_sm * 128;
    m->host_chunk = m->cap < two_waves ? m->cap : two_waves;
    const int64_t f_seq = has_seq(m) ? 4 * T : 0, f_sig = has_signal(m) ? (int64_t)T * S : 0;
    const size_t in_bytes = sizeof(float) * m->host_chunk * (f_seq + f_sig);
    const size_t out_bytes = m->host_chunk * (sizeof(float) * 2 * C + sizeof(int32_t));
    DSP_CUDA(cudaStreamCreateWithFlags(&m->copy_stream, cudaStreamNonBlocking));
    DSP_CUDA(cudaStreamCreateWithFlags(&m->compute_stream, cudaStreamNonBlocking));
    DSP_CUDA(cudaStreamCreateWithFlags(&m->d2h_stream, cudaStreamNonBlocking));
    for (int i = 0; i < Model::NBUF; ++i) {
        DSP_CUDA(cudaMalloc(&m->dev_in[i], in_bytes));
        DSP_CUDA(cudaMalloc(&m->dev_out[i], out_bytes));
        DSP_CUDA(cudaEventCreateWithFlags(&m->ev_h2d[i], cudaEventDisableTiming));
        DSP_CUDA(cudaEventCreateWithFlags(&m->ev_done[i], cudaEventDisableTiming));
        DSP_CUDA(cudaEventCreateWithFlags(&m->ev_computed[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < Model::NTICKET; ++i) DSP_CUDA(cudaEventCreateWithFlags(&m->ev_ticket[i], cudaEventDisableTiming));
    return DSP_OK;
}

static int host_check_args(Model* m, const char* who, const float* kmer, const float* base_means, const float* base_stds,
                           const float* base_signal_lens, const float* signals, int64_t n, float* logits, float* probs) {
    DSP_REQUIRE(m->packed, DSP_ERR_STATE, "%s: weights not packed", who);
    DSP_REQUIRE(n >= 0, DSP_ERR_INVALID, "%s: negative batch", who);
    if (n == 0) return DSP_OK;
    DSP_REQUIRE(logits && probs, DSP_ERR_INVALID, "%s: null output pointer", who);
    if (has_seq(m)) DSP_REQUIRE(kmer && base_means && base_stds && base_signal_lens, DSP_ERR_INVALID,
                                "%s: sequence features are required for this module", who);
    if (has_signal(m)) DSP_REQUIRE(signals, DSP_ERR_INVALID, "%s: signals are required for this module", who);
    return DSP_OK;
}

// enqueue all chunks of one batch; blocking == false requires direct (pinned) inputs and outputs
static int host_enqueue(Model* m, const float* kmer, const float* base_means, const float* base_stds,
                        const float* base_signal_lens, const float* signals, uint64_t seed, int64_t n,
                        float* logits, float* probs, int32_t* labels, bool direct_in, bool direct_out) {
    const dsp_config& c = m->cfg;
    const int T = c.seq_len, S = c.signal_len, C = c.num_classes;
    const int64_t hc = m->host_chunk;
    const int64_t f_seq = has_seq(m) ? 4 * T : 0, f_sig = has_signal(m) ? (int64_t)T * S : 0;
    const size_t in_bytes = sizeof(float) * hc * (f_seq + f_sig);
    const size_t out_bytes = hc * (sizeof(float) * 2 * C + sizeof(int32_t));
    if (m->timing) { m->spans.clear(); m->event_next = 0; }
    const int64_t nchunks = (n + hc - 1) / hc;
    struct Pending { int64_t s, cn; int b; bool live; } pend[Model::NBUF] = {};
    auto drain = [&](Pending& pd) -> int {       // staged results of one chunk -> caller memory
        if (!pd.live) return DSP_OK;
        DSP_CUDA(cudaEventSynchronize(m->ev_done[pd.b]));
        const char* po = (const char*)m->pinned_out[pd.b];
        memcpy(logits + pd.s * C, po, sizeof(float) * pd.cn * C);
        memcpy(probs + pd.s * C, po + sizeof(float) * hc * C, sizeof(float) * pd.cn * C);
        if (labels) memcpy(labels + pd.s, po + sizeof(float) * hc * 2 * C, sizeof(int32_t) * pd.cn);
        pd.live = false;
        return DSP_OK;
    };
    for (int64_t ci = 0; ci < nchunks; ++ci) {
        const int b = (int)(m->host_chunks_enqueued++ % Model::NBUF);
        const int64_t s = ci * hc, cn = (n - s < hc) ? (n - s) : hc;
        if (!direct_out) { int rc = drain(pend[b]); if (rc) return rc; }
        // the device buffers of slot b are free once the chunk that used them last has finished
        DSP_CUDA(cudaStreamWaitEvent(m->copy_stream, m->ev_done[b], 0));
        float* din = (float*)m->dev_in[b];
        float* d_kmer = din, *d_means = din + hc * T, *d_stds = din + 2 * hc * T, *d_lens = din + 3 * hc * T;
        float* d_sig = din + hc * f_seq;
        const float* src[5] = {kmer, base_means, base_stds, base_signal_lens, signals};
        float* dst[5] = {d_kmer, d_means, d_stds, d_lens, d_sig};
        const int64_t per[5] = {T, T, T, T, (int64_t)T * S};
        if (!direct_in) {
            if (!m->pinned_in[b]) DSP_CUDA(cudaMallocHost(&m->pinned_in[b], in_bytes));
            DSP_CUDA(cudaEventSynchronize(m->ev_h2d[b]));          // previous copy out of this staging buffer is done
        }
        for (int a = 0; a < 5; ++a) {
            const bool used = (a < 4) ? has_seq(m) : has_signal(m);
            if (!used) continue;
            const float* from = src[a] + s * per[a];
            if (!direct_in) {
                float* stage = (float*)m->pinned_in[b] + (dst[a] - din);
                memcpy(stage, from, sizeof(float) * cn * per[a]);
                from = stage;
            }
            DSP_CUDA(cudaMemcpyAsync(dst[a], from, sizeof(float) * cn * per[a], cudaMemcpyHostToDevice, m->copy_stream));
        }
        DSP_CUDA(cudaEventRecord(m->ev_h2d[b], m->copy_stream));
        DSP_CUDA(cudaStreamWaitEvent(m->compute_stream, m->ev_h2d[b], 0));
        char* dout = (char*)m->dev_out[b];
        float* d_logits = (float*)dout;
        float* d_probs = (float*)(dout + sizeof(float) * hc * C);
        int32_t* d_labels = (int32_t*)(dout + sizeof(float) * hc * 2 * C);
        int rc = forward_chunk(m, d_kmer, d_means, d_stds, d_lens, d_sig, nullptr, nullptr, seed, (uint64_t)ci, cn,
                               d_logits, d_probs, d_labels, m->compute_stream);
        if (rc) return rc;
        // results leave on their own stream: the device->host copies of chunk i run under chunk i+1's kernels instead
        // of in front of them
        DSP_CUDA(cudaEventRecord(m->ev_computed[b], m->compute_stream));
        DSP_CUDA(cudaStreamWaitEvent(m->d2h_stream, m->ev_computed[b], 0));
        if (direct_out) {
            DSP_CUDA(cudaMemcpyAsync(logits + s * C, d_logits, sizeof(float) * cn * C, cudaMemcpyDeviceToHost, m->d2h_stream));
            DSP_CUDA(cudaMemcpyAsync(probs + s * C, d_probs, sizeof(float) * cn * C, cudaMemcpyDeviceToHost, m->d2h_stream));
            if (labels) DSP_CUDA(cudaMemcpyAsync(labels + s, d_labels, sizeof(int32_t) * cn, cudaMemcpyDeviceToHost, m->d2h_stream));
        } else {
            if (!m->pinned_out[b]) DSP_CUDA(cudaMallocHost(&m->pinned_out[b], out_bytes));
            DSP_CUDA(cudaMemcpyAsync(m->pinned_out[b], dout, out_bytes, cudaMemcpyDeviceToHost, m->d2h_stream));
            pend[b] = {s, cn, b, true};
        }
        DSP_CUDA(cudaEventRecord(m->ev_done[b], m->d2h_stream));
    }
    if (!direct_out) for (int b = 0; b < Model::NBUF; ++b) { int rc = drain(pend[b]); if (rc) return rc; }
    return DSP_OK;
}

int dsp_forward_host(dsp_handle h, const float* kmer, const float* base_means, const float* base_stds,
                     const float* base_signal_lens, const float* signals, uint64_t seed, int64_t n,
                     float* logits, float* probs, int32_t* labels) {
    DSP_REQUIRE(h, DSP_ERR_INVALID, "dsp_forward_host: null handle");
    Model* m = h;
    int rc = host_check_args(m, "dsp_forward_host", kmer, base_means, base_stds, base_signal_lens, signals, n, logits, probs);
    if (rc || n == 0) return rc;
    DeviceGuard guard(m->cfg.device);
    if ((rc = host_setup(m))) return rc;
    const bool direct_in = (!has_seq(m) || (is_device_accessible_host(kmer) && is_device_accessible_host(base_means) &&
                                            is_device_accessible_host(base_stds) && is_device_accessible_host(base_signal_lens))) &&
                           (!has_signal(m) || is_device_accessible_host(signals));
    const bool direct_out = is_device_accessible_host(logits) && is_device_accessible_host(probs) &&
                            (!labels || is_device_accessible_host(labels));
    if ((rc = host_enqueue(m, kmer, base_means, base_stds, base_signal_lens, signals, seed, n, logits, probs, labels,
                           direct_in, direct_out))) return rc;
    DSP_CUDA(cudaStreamSynchronize(m->d2h_stream));      // every chunk's results were copied out (in order) on this stream
    return DSP_OK;
}

int dsp_forward_host_submit(dsp_handle h, const float* kmer, const float* base_means, const float* base_stds,
                            const float* base_signal_lens, const float* signals, uint64_t seed, int64_t n,
                            float* logits, float* probs, int32_t* labels, int64_t* ticket) {
    DSP_REQUIRE(h && ticket, DSP_ERR_INVALID, "dsp_forward_host_submit: null argument");
    Model* m = h;
    int rc = host_check_args(m, "dsp_forward_host_submit", kmer, base_means, base_stds, base_signal_lens, signals, n, logits, probs);
    if (rc) return rc;
    DeviceGuard guard(m->cfg.device);
    if ((rc = host_setup(m))) return rc;
    const bool direct = (!has_seq(m) || (is_device_accessible_host(kmer) && is_device_accessible_host(base_means) &&
                                         is_device_accessible_host(base_stds) && is_device_accessible_host(base_signal_lens))) &&
                        (!has_signal(m) || is_device_accessible_host(signals)) &&
                        (n == 0 || (is_device_accessible_host(logits) && is_device_accessible_host(probs) &&
                                    (!labels || is_device_accessible_host(labels))));
    DSP_REQUIRE(direct, DSP_ERR_INVALID,
                "dsp_forward_host_submit: every host buffer must be page-locked (cudaHostAlloc / cudaHostRegister / "
                "torch pin_memory); use dsp_forward_host for pageable memory");
    if (n > 0 && (rc = host_enqueue(m, kmer, base_means, base_stds, base_signal_lens, signals, seed, n, logits, probs, labels,
                                    true, true))) return rc;
    const uint64_t t = m->tickets_issued++;
    DSP_CUDA(cudaEventRecord(m->ev_ticket[t % Model::NTICKET], m->d2h_stream));   // after the last chunk's copies (n == 0: after all earlier work)
    *ticket = (int64_t)t;
    return DSP_OK;
}

int dsp_forward_host_wait(dsp_handle h, int64_t ticket) {
    DSP_REQUIRE(h, DSP_ERR_INVALID, "dsp_forward_host_wait: null handle");
    Model* m = h;
    DSP_REQUIRE(ticket >= 0 && (uint64_t)ticket < m->tickets_issued, DSP_ERR_INVALID, "dsp_forward_host_wait: unknown ticket");
    DeviceGuard guard(m->cfg.device);
    if ((uint64_t)ticket + Model::NTICKET <= m->tickets_issued) {
        // its event slot was re-used by a later submission on the same stream: that one finishing implies this one did
        DSP_CUDA(cudaEventSynchronize(m->ev_ticket[(m->tickets_issued - 1) % Model::NTICKET]));
        return DSP_OK;
    }
    DSP_CUDA(cudaEventSynchronize(m->ev_ticket[(uint64_t)ticket % Model::NTICKET]));
    return DSP_OK;
}

int dsp_train_shape(dsp_handle h, int32_t* n_params, int32_t* n_masks) {
    DSP_REQUIRE(h, DSP_ERR_INVALID, "dsp_train_shape: null handle");
    return train_shape(h, n_params, n_masks);
}

int64_t dsp_train_arena_bytes(dsp_handle h, int64_t n) { return (h && n >= 0) ? train_arena_bytes(h, n) : -1; }
int64_t dsp_train_workspace_bytes(dsp_handle h, int64_t n) { return (h && n >= 0) ? train_workspace_bytes(h, n) : -1; }

// Everything the training entries refuse before a launch; tables as in include/dsp_b200.h.
static int train_check(Model* m, const char* who, int G, const float* const* params, int32_t n_params,
                       const float* const* masks, const void* const* arenas, int64_t n) {
    int32_t np = 0, nm = 0;
    train_shape(m, &np, &nm);
    DSP_REQUIRE(G >= 1 && G <= DSP_TRAIN_MAX_MODELS, DSP_ERR_INVALID, "%s: %d models, must be 1..%d", who, G,
                DSP_TRAIN_MAX_MODELS);
    DSP_REQUIRE(params && masks && arenas, DSP_ERR_INVALID, "%s: null argument", who);
    DSP_REQUIRE(n_params == np, DSP_ERR_INVALID, "%s: %d parameters given, this configuration has %d", who, n_params, np);
    for (int i = 0; i < G * np; ++i)
        DSP_REQUIRE(params[i], DSP_ERR_INVALID, "%s: parameter %d of model %d is null", who, i % np, i / np);
    for (int i = 0; i < G; ++i) DSP_REQUIRE(arenas[i], DSP_ERR_INVALID, "%s: arena of model %d is null", who, i);
    for (int i = 1; i < G; ++i)
        for (int k = 0; k < nm; ++k)
            DSP_REQUIRE(!masks[i * nm + k] == !masks[k], DSP_ERR_INVALID,
                        "%s: dropout mask slot %d is null for some models and not for others", who, k);
    DSP_REQUIRE(n >= 1, DSP_ERR_INVALID, "%s: batch must hold at least one site", who);
    return DSP_OK;
}

static int train_forward_checked(Model* m, const char* who, int G, const float* const* params, int32_t n_params,
                                 const float* const* inputs, const float* const* states, const uint64_t* seeds,
                                 const float* const* masks, int64_t n, void* const* arenas, float* const* logits,
                                 void* stream) {
    int rc = train_check(m, who, G, params, n_params, masks, arenas, n);
    if (rc) return rc;
    DSP_REQUIRE(inputs && seeds && logits, DSP_ERR_INVALID, "%s: null argument", who);
    for (int i = 0; i < G; ++i) {
        const float* const* in = inputs + 5 * i;
        DSP_REQUIRE(logits[i], DSP_ERR_INVALID, "%s: null output pointer (model %d)", who, i);
        if (has_seq(m)) DSP_REQUIRE(in[0] && in[1] && in[2] && in[3], DSP_ERR_INVALID,
                                    "%s: sequence features are required for this module (model %d)", who, i);
        if (has_signal(m)) DSP_REQUIRE(in[4], DSP_ERR_INVALID, "%s: signals are required for this module (model %d)", who, i);
        if (states)
            for (int g = 0; g < 3; ++g) {
                if ((g == 0 && !has_seq(m)) || (g == 1 && !has_signal(m))) continue;
                DSP_REQUIRE(states[6 * i + 2 * g] && states[6 * i + 2 * g + 1], DSP_ERR_INVALID,
                            "%s: states[%d] of model %d is null", who, 2 * g, i);
            }
    }
    DeviceGuard guard(m->cfg.device);
    return train_forward(m, G, params, inputs, states, seeds, masks, n, arenas, logits, (cudaStream_t)stream);
}

static int train_backward_checked(Model* m, const char* who, int G, const float* const* params, int32_t n_params,
                                  const float* const* masks, const void* const* arenas, const float* const* dlogits,
                                  int64_t n, void* const* workspaces, float* const* grads, void* stream) {
    int rc = train_check(m, who, G, params, n_params, masks, arenas, n);
    if (rc) return rc;
    DSP_REQUIRE(dlogits && workspaces && grads, DSP_ERR_INVALID, "%s: null argument", who);
    for (int i = 0; i < G; ++i)
        DSP_REQUIRE(dlogits[i] && workspaces[i], DSP_ERR_INVALID, "%s: null argument (model %d)", who, i);
    for (int i = 0; i < G * n_params; ++i)
        DSP_REQUIRE(grads[i], DSP_ERR_INVALID, "%s: gradient %d of model %d is null", who, i % n_params, i / n_params);
    DeviceGuard guard(m->cfg.device);
    return train_backward(m, G, params, masks, arenas, dlogits, n, workspaces, grads, (cudaStream_t)stream);
}

int dsp_train_forward(dsp_handle h, const float* const* params, int32_t n_params, const float* kmer,
                      const float* base_means, const float* base_stds, const float* base_signal_lens,
                      const float* signals, const float* const* states, uint64_t seed,
                      const float* const* dropout_masks, int64_t n, void* arena, float* logits, void* stream) {
    DSP_REQUIRE(h, DSP_ERR_INVALID, "dsp_train_forward: null handle");
    const float* inputs[5] = {kmer, base_means, base_stds, base_signal_lens, signals};
    return train_forward_checked(h, "dsp_train_forward", 1, params, n_params, inputs, states, &seed, dropout_masks, n,
                                 &arena, &logits, stream);
}

int dsp_train_backward(dsp_handle h, const float* const* params, int32_t n_params, const float* const* dropout_masks,
                       const void* arena, const float* dlogits, int64_t n, void* workspace, float* const* grads,
                       void* stream) {
    DSP_REQUIRE(h, DSP_ERR_INVALID, "dsp_train_backward: null handle");
    return train_backward_checked(h, "dsp_train_backward", 1, params, n_params, dropout_masks, &arena, &dlogits, n,
                                  &workspace, grads, stream);
}

int dsp_train_forward_batch(dsp_handle h, int32_t n_models, const float* const* params, int32_t n_params,
                            const float* const* inputs, const float* const* states, const uint64_t* seeds,
                            const float* const* dropout_masks, int64_t n, void* const* arenas,
                            float* const* logits, void* stream) {
    DSP_REQUIRE(h, DSP_ERR_INVALID, "dsp_train_forward_batch: null handle");
    return train_forward_checked(h, "dsp_train_forward_batch", n_models, params, n_params, inputs, states, seeds,
                                 dropout_masks, n, arenas, logits, stream);
}

int dsp_train_backward_batch(dsp_handle h, int32_t n_models, const float* const* params, int32_t n_params,
                             const float* const* dropout_masks, const void* const* arenas,
                             const float* const* dlogits, int64_t n, void* const* workspaces,
                             float* const* grads, void* stream) {
    DSP_REQUIRE(h, DSP_ERR_INVALID, "dsp_train_backward_batch: null handle");
    return train_backward_checked(h, "dsp_train_backward_batch", n_models, params, n_params, dropout_masks, arenas,
                                  dlogits, n, workspaces, grads, stream);
}

int64_t dsp_launch_count(dsp_handle h) { return h ? h->launches : 0; }

int dsp_set_timing(dsp_handle h, int enable) {
    DSP_REQUIRE(h, DSP_ERR_INVALID, "dsp_set_timing: null handle");
    h->timing = enable != 0;
    h->spans.clear();
    h->event_next = 0;
    return DSP_OK;
}

int dsp_get_timing(dsp_handle h, int which, float* ms, int64_t* launches) {
    DSP_REQUIRE(h && ms, DSP_ERR_INVALID, "dsp_get_timing: null argument");
    DeviceGuard guard(h->cfg.device);
    float total = 0.f;
    int64_t cnt = 0;
    for (const TimingSpan& s : h->spans) {
        if (s.cls != which) continue;
        DSP_CUDA(cudaEventSynchronize(s.b));
        float t = 0.f;
        DSP_CUDA(cudaEventElapsedTime(&t, s.a, s.b));
        total += t;
        ++cnt;
    }
    *ms = total;
    if (launches) *launches = cnt;
    return DSP_OK;
}

}  // extern "C"
