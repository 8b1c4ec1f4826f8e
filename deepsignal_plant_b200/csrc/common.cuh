// Shared internal declarations of libdsp_b200 (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <string>
#include <vector>
#include <map>
#include "../../include/dsp_b200.h"

namespace dsp {

void set_error(const char* fmt, ...);

#define DSP_CUDA(call)                                                                   \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess) {                                                        \
            dsp::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call,                 \
                           cudaGetErrorString(e__));                                     \
            return DSP_ERR_CUDA;                                                         \
        }                                                                                \
    } while (0)

#define DSP_REQUIRE(cond, status, ...)                                                   \
    do {                                                                                 \
        if (!(cond)) {                                                                   \
            dsp::set_error(__VA_ARGS__);                                                 \
            return (status);                                                             \
        }                                                                                \
    } while (0)

static inline int ru(int x, int m) { return (x + m - 1) / m * m; }

// One direction of one LSTM layer in the fp32 kernel layout.
//   wt: [(Kp + Hp)][4][H] float, row k = input feature (x part first, zero padded to
//       Kp = ru(K,4), then the recurrent part padded to Hp = ru(H,4)), then gate
//       (i,f,g,o), then hidden unit -- so that consecutive threads (= hidden units)
//       read consecutive floats.
//   bias: [4][H] = bias_ih + bias_hh.
struct LstmDirF32 {
    float* wt = nullptr;
    float* bias = nullptr;
};

struct LstmLayer {
    int K = 0, H = 0;
    LstmDirF32 f32[2];
    // FP16 tensor-core layout (kernels_tc.cu): see TcLayerPack there.
    void* tc = nullptr;
};

// A dense layer y = act(W x + b) in the fp32 kernel layout: wt [Kp][J], bias [J].
struct DenseF32 {
    int K = 0, J = 0;
    float* wt = nullptr;
    float* bias = nullptr;
    void* tc = nullptr;
};

struct TimingSpan {
    int cls;
    cudaEvent_t a, b;
};

struct Model {
    dsp_config cfg;
    int nhid_seq = 0, nhid_signal = 0, kseq = 0;
    bool packed = false;
    std::map<std::string, std::vector<float>> params;   // host copies until packed

    float* embed = nullptr;                 // [vocab][E] fp32
    std::vector<LstmLayer> lstm_seq, lstm_signal, lstm_comb;
    DenseF32 fc_seq, fc_signal, fc1, fc2;

    // workspace for cfg.max_batch sites
    int64_t cap = 0;
    float* xseq = nullptr;                  // (cap, T, kseq)
    float* buf[2] = {nullptr, nullptr};     // (cap, T, 2*Hmax) ping-pong
    float* comb_in = nullptr;               // (cap, T, hidden)
    float* states = nullptr;                // Philox-drawn initial states
    int64_t state_floats_per_site = 0;
    std::vector<void*> device_allocs;       // workspace first, then the packed-weight arena
    size_t n_workspace_allocs = 0;          // device_allocs[0 .. n_workspace_allocs) survive a re-pack

    // host staging for dsp_forward_host
    cudaStream_t copy_stream = nullptr, compute_stream = nullptr, d2h_stream = nullptr;
    static constexpr int NBUF = 3;          // chunks in flight: copy in / compute / copy out
    static constexpr int NTICKET = 8;
    void* pinned_in[NBUF] = {};             // staging for pageable caller memory (lazily allocated)
    void* pinned_out[NBUF] = {};
    void* dev_in[NBUF] = {};
    void* dev_out[NBUF] = {};
    cudaEvent_t ev_h2d[NBUF] = {}, ev_done[NBUF] = {}, ev_computed[NBUF] = {};
    cudaEvent_t ev_ticket[NTICKET] = {};
    int64_t host_chunk = 0;                 // sites per staged chunk (two full waves of CTA pairs)
    uint64_t host_chunks_enqueued = 0;      // buffer ring position, carried across calls
    uint64_t tickets_issued = 0;
    int n_sm = 0;

    int64_t launches = 0;
    bool timing = false;
    std::vector<TimingSpan> spans;
    std::vector<cudaEvent_t> event_pool;
    size_t event_next = 0;

    void* tc_state = nullptr;               // owned by kernels_tc.cu
};

inline cudaEvent_t next_event(Model* m) {
    if (m->event_next == m->event_pool.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        m->event_pool.push_back(e);
    }
    return m->event_pool[m->event_next++];
}

// CUDA-event bracket around the launches of one kernel class (dsp_set_timing / dsp_get_timing).
struct Span {
    Model* m; cudaStream_t st; cudaEvent_t a = nullptr;
    int cls;
    Span(Model* m_, int cls_, cudaStream_t st_) : m(m_), st(st_), cls(cls_) {
        if (m->timing) { a = next_event(m); cudaEventRecord(a, st); }
    }
    ~Span() {
        if (m->timing) { cudaEvent_t b = next_event(m); cudaEventRecord(b, st); m->spans.push_back({cls, a, b}); }
    }
};

// ---- fp32 CUDA-core path (kernels_f32.cu) --------------------------------------------
int f32_assemble_seq(Model* m, const float* kmer, const float* means, const float* stds,
                     const float* lens, int64_t n, float* xseq, cudaStream_t st);
int f32_lstm_layer(Model* m, const LstmLayer& L, const float* x, int x_row_stride, int x_t_stride,
                   const float* h0, const float* c0, int64_t state_dir_stride,
                   float* y, int64_t n, cudaStream_t st);
int f32_dense(Model* m, const DenseF32& D, const float* x, int64_t rows, int x_row_stride,
              float* y, int y_row_stride, int relu, cudaStream_t st);
int f32_head(Model* m, const float* y_last, int64_t n, float* logits, float* probs,
             int32_t* labels, cudaStream_t st);
// same head on a flat (n, 2H) fp32 matrix [h_fwd(T-1) | h_bwd(0)]
int f32_head_flat(Model* m, const float* hfinal, int64_t n, float* logits, float* probs,
                  int32_t* labels, cudaStream_t st);
int philox_normal(Model* m, float* out, int64_t count, uint64_t seed, uint64_t stream_id,
                  cudaStream_t st);

// ---- fp32 training path (kernels_train.cu) ----------------------------------------------
int train_shape(const Model* m, int32_t* n_params, int32_t* n_masks);
int64_t train_arena_bytes(const Model* m, int64_t n);
int64_t train_workspace_bytes(const Model* m, int64_t n);
int train_forward(Model* m, const float* const* params, const float* kmer, const float* means, const float* stds,
                  const float* lens, const float* signals, const float* const* states6, uint64_t seed,
                  const float* const* masks, int64_t n, void* arena, float* logits, cudaStream_t st);
int train_backward(Model* m, const float* const* params, const float* const* masks, const void* arena,
                   const float* dlogits, int64_t n, void* workspace, float* const* grads, cudaStream_t st);

}  // namespace dsp

// the opaque handle type of the C ABI
struct dsp_model_s : public dsp::Model {};
