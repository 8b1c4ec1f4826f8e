// fp32 CUDA-core kernels of the ModelBiLSTM forward (DSP_PRECISION_FP32).
//
// This is the exact-arithmetic path: every contraction is an fp32 FMA chain, the gate
// non-linearities use expf/tanhf and true division.  It is the in-repo CUDA reference the
// tensor-core path is diffed against on the GPU box and the accuracy fallback for shapes
// the tcgen05 kernels do not cover.  Reference semantics: deepsignal_plant/models.py:178-240
// (dataflow) and torch nn.LSTM (gate order i,f,g,o; reverse direction walks t = T-1..0).
#include "common.cuh"
#include <curand_kernel.h>
#include "philox.cuh"

namespace dsp {

namespace {

constexpr int TS = 16;   // sites (rows) per CTA

__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

// ---------------------------------------------------------------------------------------
// Feature assembly (models.py:182-195): [embed(kmer) | mean | std | len] per base.
__global__ void assemble_seq_kernel(const float* __restrict__ kmer, const float* __restrict__ means,
                                    const float* __restrict__ stds, const float* __restrict__ lens,
                                    const float* __restrict__ embed, int E, int vocab, int use_len,
                                    int kseq, int64_t rows, float* __restrict__ x) {
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    float* o = x + r * kseq;
    int c = 0;
    if (E > 0) {
        long long code = (long long)kmer[r];            // kmer.long(): truncation toward zero
        if (code < 0) code = 0;
        if (code >= vocab) code = vocab - 1;
        for (int e = 0; e < E; ++e) o[c++] = embed[code * E + e];
    }
    o[c++] = means[r];
    o[c++] = stds[r];
    if (use_len) o[c++] = lens[r];
}

// ---------------------------------------------------------------------------------------
// One bidirectional LSTM layer.  grid = (ceil(n/TS), 2 directions); each CTA walks its TS
// sites through all T steps of one direction.  Per step the gate pre-activations of hidden
// unit j for all TS sites are accumulated by one thread (acc[TS][4]), the weights of that
// unit streamed from L2 in a k-major layout that is coalesced across units, the activation
// rows broadcast from shared memory.
template <int TS_>
__global__ void __launch_bounds__(256, 2)
lstm_layer_f32_kernel(const float* __restrict__ x, int x_row_stride, int x_t_stride, int K,
                      const float* __restrict__ wt0, const float* __restrict__ wt1,
                      const float* __restrict__ bias0, const float* __restrict__ bias1,
                      const float* __restrict__ h0, const float* __restrict__ c0,
                      int64_t state_dir_stride, float* __restrict__ y, int H, int T, int64_t n) {
    extern __shared__ float smem[];
    const int Kp = (K + 3) & ~3, Hp = (H + 3) & ~3;
    float* ax = smem;                    // [TS][Kp]
    float* ah = ax + TS_ * Kp;           // [2][TS][Hp]
    float* cs = ah + 2 * TS_ * Hp;       // [TS][Hp]
    const int dir = blockIdx.y;
    const float* __restrict__ wt = dir ? wt1 : wt0;
    const float* __restrict__ bias = dir ? bias1 : bias0;
    const int64_t site0 = (int64_t)blockIdx.x * TS_;
    const int tid = threadIdx.x, nthr = blockDim.x;

    for (int i = tid; i < TS_ * Hp; i += nthr) {
        int s = i / Hp, j = i - s * Hp;
        int64_t site = site0 + s;
        float hv = 0.f, cv = 0.f;
        if (site < n && j < H) {
            hv = h0[dir * state_dir_stride + site * H + j];
            cv = c0[dir * state_dir_stride + site * H + j];
        }
        ah[i] = hv;
        ah[TS_ * Hp + i] = 0.f;
        cs[i] = cv;
    }
    int cur = 0;
    for (int step = 0; step < T; ++step) {
        const int t = dir ? (T - 1 - step) : step;
        for (int i = tid; i < TS_ * Kp; i += nthr) {
            int s = i / Kp, k = i - s * Kp;
            int64_t site = site0 + s;
            ax[i] = (site < n && k < K) ? x[site * x_row_stride + (int64_t)t * x_t_stride + k] : 0.f;
        }
        __syncthreads();
        const float* hprev = ah + cur * TS_ * Hp;
        float* hnext = ah + (cur ^ 1) * TS_ * Hp;
        for (int j = tid; j < H; j += nthr) {
            float acc[TS_][4];
            const float b_i = bias[j], b_f = bias[H + j], b_g = bias[2 * H + j], b_o = bias[3 * H + j];
#pragma unroll
            for (int s = 0; s < TS_; ++s) { acc[s][0] = b_i; acc[s][1] = b_f; acc[s][2] = b_g; acc[s][3] = b_o; }
            const float* w = wt + j;
            for (int k = 0; k < Kp; k += 4) {
                float wv[4][4];
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
#pragma unroll
                    for (int g = 0; g < 4; ++g) wv[kk][g] = __ldg(w + ((int64_t)(k + kk) * 4 + g) * H);
#pragma unroll
                for (int s = 0; s < TS_; ++s) {
                    const float4 a = *reinterpret_cast<const float4*>(ax + s * Kp + k);
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        acc[s][g] = fmaf(a.x, wv[0][g], acc[s][g]);
                        acc[s][g] = fmaf(a.y, wv[1][g], acc[s][g]);
                        acc[s][g] = fmaf(a.z, wv[2][g], acc[s][g]);
                        acc[s][g] = fmaf(a.w, wv[3][g], acc[s][g]);
                    }
                }
            }
            w = wt + (int64_t)Kp * 4 * H + j;
            for (int k = 0; k < Hp; k += 4) {
                float wv[4][4];
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
#pragma unroll
                    for (int g = 0; g < 4; ++g) wv[kk][g] = __ldg(w + ((int64_t)(k + kk) * 4 + g) * H);
#pragma unroll
                for (int s = 0; s < TS_; ++s) {
                    const float4 a = *reinterpret_cast<const float4*>(hprev + s * Hp + k);
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        acc[s][g] = fmaf(a.x, wv[0][g], acc[s][g]);
                        acc[s][g] = fmaf(a.y, wv[1][g], acc[s][g]);
                        acc[s][g] = fmaf(a.z, wv[2][g], acc[s][g]);
                        acc[s][g] = fmaf(a.w, wv[3][g], acc[s][g]);
                    }
                }
            }
#pragma unroll
            for (int s = 0; s < TS_; ++s) {
                const float ig = sigmoid_f(acc[s][0]);
                const float fg = sigmoid_f(acc[s][1]);
                const float gg = tanhf(acc[s][2]);
                const float og = sigmoid_f(acc[s][3]);
                const float c = fg * cs[s * Hp + j] + ig * gg;
                const float h = og * tanhf(c);
                cs[s * Hp + j] = c;
                hnext[s * Hp + j] = h;
                const int64_t site = site0 + s;
                if (site < n) y[(site * T + t) * (2 * (int64_t)H) + dir * H + j] = h;
            }
        }
        __syncthreads();
        cur ^= 1;
    }
}

// ---------------------------------------------------------------------------------------
// Dense rows: y[r][j] = act(bias[j] + sum_k x[r][k] * wt[k][j]).
template <int TS_>
__global__ void __launch_bounds__(256)
dense_f32_kernel(const float* __restrict__ x, int64_t rows, int x_row_stride, int K,
                 const float* __restrict__ wt, const float* __restrict__ bias, int J,
                 float* __restrict__ y, int y_row_stride, int relu) {
    extern __shared__ float smem[];
    const int Kp = (K + 3) & ~3;
    const int64_t r0 = (int64_t)blockIdx.x * TS_;
    for (int i = threadIdx.x; i < TS_ * Kp; i += blockDim.x) {
        int s = i / Kp, k = i - s * Kp;
        int64_t r = r0 + s;
        smem[i] = (r < rows && k < K) ? x[r * x_row_stride + k] : 0.f;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < J; j += blockDim.x) {
        float acc[TS_];
        const float b = bias[j];
#pragma unroll
        for (int s = 0; s < TS_; ++s) acc[s] = b;
        for (int k = 0; k < Kp; k += 4) {
            const float w0 = __ldg(wt + (int64_t)(k + 0) * J + j), w1 = __ldg(wt + (int64_t)(k + 1) * J + j);
            const float w2 = __ldg(wt + (int64_t)(k + 2) * J + j), w3 = __ldg(wt + (int64_t)(k + 3) * J + j);
#pragma unroll
            for (int s = 0; s < TS_; ++s) {
                const float4 a = *reinterpret_cast<const float4*>(smem + s * Kp + k);
                acc[s] = fmaf(a.x, w0, acc[s]);
                acc[s] = fmaf(a.y, w1, acc[s]);
                acc[s] = fmaf(a.z, w2, acc[s]);
                acc[s] = fmaf(a.w, w3, acc[s]);
            }
        }
#pragma unroll
        for (int s = 0; s < TS_; ++s) {
            const int64_t r = r0 + s;
            if (r < rows) y[r * y_row_stride + j] = relu ? fmaxf(acc[s], 0.f) : acc[s];
        }
    }
}

// ---------------------------------------------------------------------------------------
// Head (models.py:229-240): [fwd h(T-1) | bwd h(0)] -> fc1 -> ReLU -> fc2 -> softmax (+argmax).
template <int TS_>
__global__ void __launch_bounds__(256)
head_f32_kernel(const float* __restrict__ ylast, int H, int T, int64_t n,
                const float* __restrict__ w1t, const float* __restrict__ b1, int J1,
                const float* __restrict__ w2t, const float* __restrict__ b2, int C,
                float* __restrict__ logits, float* __restrict__ probs, int32_t* __restrict__ labels) {
    extern __shared__ float smem[];
    const int K = 2 * H;                 // multiple of 2; pad to 4
    const int Kp = (K + 3) & ~3, J1p = (J1 + 3) & ~3;
    float* in = smem;                    // [TS][Kp]
    float* z = in + TS_ * Kp;            // [TS][J1p]
    float* lg = z + TS_ * J1p;           // [TS][C]
    const int64_t r0 = (int64_t)blockIdx.x * TS_;
    for (int i = threadIdx.x; i < TS_ * Kp; i += blockDim.x) {
        int s = i / Kp, k = i - s * Kp;
        int64_t r = r0 + s;
        float v = 0.f;
        if (r < n && k < K) {
            const int t = (k < H) ? (T - 1) : 0;
            v = ylast[(r * T + t) * (int64_t)K + k];
        }
        in[i] = v;
    }
    for (int i = threadIdx.x; i < TS_ * J1p; i += blockDim.x) z[i] = 0.f;
    __syncthreads();
    for (int j = threadIdx.x; j < J1; j += blockDim.x) {
        float acc[TS_];
        const float b = b1[j];
#pragma unroll
        for (int s = 0; s < TS_; ++s) acc[s] = b;
        for (int k = 0; k < Kp; k += 4) {
            const float w0 = __ldg(w1t + (int64_t)(k + 0) * J1 + j), w1 = __ldg(w1t + (int64_t)(k + 1) * J1 + j);
            const float w2 = __ldg(w1t + (int64_t)(k + 2) * J1 + j), w3 = __ldg(w1t + (int64_t)(k + 3) * J1 + j);
#pragma unroll
            for (int s = 0; s < TS_; ++s) {
                const float4 a = *reinterpret_cast<const float4*>(in + s * Kp + k);
                acc[s] = fmaf(a.x, w0, acc[s]);
                acc[s] = fmaf(a.y, w1, acc[s]);
                acc[s] = fmaf(a.z, w2, acc[s]);
                acc[s] = fmaf(a.w, w3, acc[s]);
            }
        }
#pragma unroll
        for (int s = 0; s < TS_; ++s) z[s * J1p + j] = fmaxf(acc[s], 0.f);
    }
    __syncthreads();
    // fc2: one warp per (site, class) pair, strided
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    for (int p = warp; p < TS_ * C; p += nwarp) {
        const int s = p / C, c = p - s * C;
        float acc = 0.f;
        for (int k = lane; k < J1; k += 32) acc = fmaf(z[s * J1p + k], __ldg(w2t + (int64_t)k * C + c), acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) lg[p] = acc + b2[c];
    }
    __syncthreads();
    for (int s = threadIdx.x; s < TS_; s += blockDim.x) {
        const int64_t r = r0 + s;
        if (r >= n) continue;
        float mx = lg[s * C];
        int arg = 0;
        for (int c = 1; c < C; ++c) if (lg[s * C + c] > mx) { mx = lg[s * C + c]; arg = c; }
        float sum = 0.f;
        for (int c = 0; c < C; ++c) sum += expf(lg[s * C + c] - mx);
        for (int c = 0; c < C; ++c) {
            logits[r * C + c] = lg[s * C + c];
            probs[r * C + c] = expf(lg[s * C + c] - mx) / sum;
        }
        if (labels) labels[r] = arg;
    }
}

// ---------------------------------------------------------------------------------------
// N(0,1) initial states: philox_normal_quad (philox.cuh), one thread per group of four outputs.
__global__ void philox_normal_kernel(float* __restrict__ out, int64_t count, uint64_t seed,
                                     uint64_t stream_id) {
    philox_normal_quad(out, count, seed, stream_id, (int64_t)blockIdx.x * blockDim.x + threadIdx.x);
}

}  // namespace

int f32_assemble_seq(Model* m, const float* kmer, const float* means, const float* stds,
                     const float* lens, int64_t n, float* xseq, cudaStream_t st) {
    const dsp_config& c = m->cfg;
    int64_t rows = n * c.seq_len;
    if (rows == 0) return DSP_OK;
    int E = c.is_base ? c.embedding_size : 0;
    assemble_seq_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(
        kmer, means, stds, lens, m->embed, E, c.vocab_size, c.is_signallen, m->kseq, rows, xseq);
    m->launches++;
    DSP_CUDA(cudaGetLastError());
    return DSP_OK;
}

int f32_lstm_layer(Model* m, const LstmLayer& L, const float* x, int x_row_stride, int x_t_stride,
                   const float* h0, const float* c0, int64_t state_dir_stride,
                   float* y, int64_t n, cudaStream_t st) {
    if (n == 0) return DSP_OK;
    const int Kp = ru(L.K, 4), Hp = ru(L.H, 4);
    size_t smem = sizeof(float) * TS * (size_t)(Kp + 3 * Hp);
    DSP_REQUIRE(smem <= 227 * 1024, DSP_ERR_INVALID, "fp32 LSTM layer K=%d H=%d exceeds shared memory", L.K, L.H);
    DSP_CUDA(cudaFuncSetAttribute(lstm_layer_f32_kernel<TS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024)));
    int threads = L.H >= 256 ? 256 : ru(L.H, 32);
    dim3 grid((unsigned)((n + TS - 1) / TS), 2);
    lstm_layer_f32_kernel<TS><<<grid, threads, smem, st>>>(
        x, x_row_stride, x_t_stride, L.K, L.f32[0].wt, L.f32[1].wt, L.f32[0].bias, L.f32[1].bias,
        h0, c0, state_dir_stride, y, L.H, m->cfg.seq_len, n);
    m->launches++;
    DSP_CUDA(cudaGetLastError());
    return DSP_OK;
}

int f32_dense(Model* m, const DenseF32& D, const float* x, int64_t rows, int x_row_stride,
              float* y, int y_row_stride, int relu, cudaStream_t st) {
    if (rows == 0) return DSP_OK;
    size_t smem = sizeof(float) * TS * (size_t)ru(D.K, 4);
    DSP_REQUIRE(smem <= 48 * 1024, DSP_ERR_INVALID, "dense layer K=%d too wide", D.K);
    int threads = D.J >= 256 ? 256 : ru(D.J, 32);
    dense_f32_kernel<TS><<<(unsigned)((rows + TS - 1) / TS), threads, smem, st>>>(
        x, rows, x_row_stride, D.K, D.wt, D.bias, D.J, y, y_row_stride, relu);
    m->launches++;
    DSP_CUDA(cudaGetLastError());
    return DSP_OK;
}

static int head_launch(Model* m, const float* y_last, int T, int64_t n, float* logits, float* probs,
                       int32_t* labels, cudaStream_t st);

int f32_head(Model* m, const float* y_last, int64_t n, float* logits, float* probs,
             int32_t* labels, cudaStream_t st) {
    return head_launch(m, y_last, m->cfg.seq_len, n, logits, probs, labels, st);
}

int f32_head_flat(Model* m, const float* hfinal, int64_t n, float* logits, float* probs,
                  int32_t* labels, cudaStream_t st) {
    return head_launch(m, hfinal, 1, n, logits, probs, labels, st);     // T = 1: row r is (r, 2H)
}

static int head_launch(Model* m, const float* y_last, int T, int64_t n, float* logits, float* probs,
                       int32_t* labels, cudaStream_t st) {
    if (n == 0) return DSP_OK;
    const dsp_config& c = m->cfg;
    const int H = c.hidden_size, J1 = m->fc1.J, C = c.num_classes;
    size_t smem = sizeof(float) * TS * (size_t)(ru(2 * H, 4) + ru(J1, 4) + C);
    DSP_REQUIRE(smem <= 227 * 1024, DSP_ERR_INVALID, "head too wide for shared memory");
    DSP_CUDA(cudaFuncSetAttribute(head_f32_kernel<TS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 * 1024)));
    head_f32_kernel<TS><<<(unsigned)((n + TS - 1) / TS), 256, smem, st>>>(
        y_last, H, T, n, m->fc1.wt, m->fc1.bias, J1, m->fc2.wt, m->fc2.bias, C, logits, probs, labels);
    m->launches++;
    DSP_CUDA(cudaGetLastError());
    return DSP_OK;
}

int philox_normal(Model* m, float* out, int64_t count, uint64_t seed, uint64_t stream_id,
                  cudaStream_t st) {
    if (count == 0) return DSP_OK;
    int64_t quads = (count + 3) / 4;
    philox_normal_kernel<<<(unsigned)((quads + 255) / 256), 256, 0, st>>>(out, count, seed, stream_id);
    m->launches++;
    DSP_CUDA(cudaGetLastError());
    return DSP_OK;
}

}  // namespace dsp
