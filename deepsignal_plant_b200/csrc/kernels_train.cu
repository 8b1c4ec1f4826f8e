// fp32 CUDA-core training path of ModelBiLSTM: forward with saved activations, backward,
// weights taken as device pointers in state_dict order (dsp_train_forward / dsp_train_backward).
//
// Reference semantics: deepsignal_plant/models.py:178-240 in train() mode -- nn.LSTM inter-layer
// dropout on every layer's output but the last of a stack, dropout -> fc1 -> dropout -> ReLU -> fc2 in
// the head, no dropout on the branch fc layers.  Dropout masks are inputs (already scaled by 1/(1-p)).
//
// The recurrent part of each LSTM layer's backward is one kernel per layer (grid: site tiles x 2
// directions) that walks time backwards and writes the pre-activation gradients dZ; every weight
// contraction is a time-batched GEMM over all n*T rows (gemm_f32_kernel).  Sums over sites are
// split-K with a fixed split count and a second, fixed-order reduction pass: no float atomics, so a
// repeated backward is bit-identical.
#include "common.cuh"
#include <algorithm>
#include <array>

namespace dsp {

namespace {

constexpr int TS = 16;   // sites (rows) per CTA of the recurrent kernels

__device__ __forceinline__ float sigmoid_t(float x) { return 1.0f / (1.0f + expf(-x)); }

// torch layout (W_ih [4H][K], W_hh [4H][H], b_ih, b_hh) -> the fp32 forward layout of common.cuh
// (wt [(Kp + Hp)][4][H], bias [4H] = b_ih + b_hh).
__global__ void repack_lstm_kernel(const float* __restrict__ wih, const float* __restrict__ whh,
                                   const float* __restrict__ bih, const float* __restrict__ bhh,
                                   int K, int H, float* __restrict__ wt, float* __restrict__ bias) {
    const int Kp = (K + 3) & ~3, Hp = (H + 3) & ~3;
    const int64_t total = (int64_t)(Kp + Hp) * 4 * H;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int row = (int)(idx / (4 * H));
        const int g = (int)((idx / H) % 4), j = (int)(idx % H);
        float v;
        if (row < Kp) v = row < K ? wih[(int64_t)(g * H + j) * K + row] : 0.f;
        else v = (row - Kp) < H ? whh[(int64_t)(g * H + j) * H + (row - Kp)] : 0.f;
        wt[idx] = v;
        if (idx < 4 * H) bias[idx] = bih[idx] + bhh[idx];
    }
}

// Feature assembly (models.py:182-195) that also keeps the embedding codes it gathered.
__global__ void assemble_seq_train_kernel(const float* __restrict__ kmer, const float* __restrict__ means,
                                          const float* __restrict__ stds, const float* __restrict__ lens,
                                          const float* __restrict__ embed, int E, int vocab, int use_len,
                                          int kseq, int64_t rows, float* __restrict__ x, int32_t* __restrict__ codes) {
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    float* o = x + r * kseq;
    int c = 0;
    long long code = (long long)kmer[r];                // kmer.long(): truncation toward zero
    if (code < 0) code = 0;
    if (code >= vocab) code = vocab - 1;
    codes[r] = (int32_t)code;
    for (int e = 0; e < E; ++e) o[c++] = embed[code * E + e];
    o[c++] = means[r];
    o[c++] = stds[r];
    if (use_len) o[c++] = lens[r];
}

// lstm_layer_f32_kernel (kernels_f32.cu) plus the saved activations of backward: the post-activation
// gates i, f, g, o at gates[((site*T + t)*2 + dir)*4H + gate*H + j] and the cell state c_t at
// cst[((site*T + t)*2 + dir)*H + j].
template <int TS_>
__global__ void __launch_bounds__(256, 2)
lstm_train_fwd_kernel(const float* __restrict__ x, int x_row_stride, int x_t_stride, int K,
                      const float* __restrict__ wt0, const float* __restrict__ wt1,
                      const float* __restrict__ bias0, const float* __restrict__ bias1,
                      const float* __restrict__ h0, const float* __restrict__ c0,
                      int64_t state_dir_stride, float* __restrict__ y, float* __restrict__ gates,
                      float* __restrict__ cst, int H, int T, int64_t n) {
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
                const float ig = sigmoid_t(acc[s][0]);
                const float fg = sigmoid_t(acc[s][1]);
                const float gg = tanhf(acc[s][2]);
                const float og = sigmoid_t(acc[s][3]);
                const float c = fg * cs[s * Hp + j] + ig * gg;
                const float h = og * tanhf(c);
                cs[s * Hp + j] = c;
                hnext[s * Hp + j] = h;
                const int64_t site = site0 + s;
                if (site < n) {
                    const int64_t rd = (site * T + t) * 2 + dir;
                    y[(site * T + t) * (2 * (int64_t)H) + dir * H + j] = h;
                    float* gp = gates + rd * 4 * H + j;
                    gp[0] = ig; gp[H] = fg; gp[2 * H] = gg; gp[3 * H] = og;
                    cst[rd * H + j] = c;
                }
            }
        }
        __syncthreads();
        cur ^= 1;
    }
}

// Recurrent part of one bidirectional LSTM layer's backward.  grid = (ceil(n/TS), 2 directions).
// Walks the direction's time order backwards with dh_rec and dc of the site tile in shared memory:
//   dh = dY[t] + dh_rec;  dc += dh*o*(1 - tanh^2 c);  dz = (dc*g*i(1-i), dc*c_prev*f(1-f), dc*i(1-g^2),
//   dh*tanh(c)*o(1-o));  dc *= f;  dh_rec = W_hh^T dz.
// Writes dz to dz[((site*T + t)*2 + dir)*4H + gate*H + j] and h_{t-1} (the previous output in the
// direction's order, h0 at its first step) to hprev[(site*T + t)*2H + dir*H + j] for dW_hh.
template <int TS_>
__global__ void __launch_bounds__(256)
lstm_train_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ gates, const float* __restrict__ cst,
                      const float* __restrict__ y, const float* __restrict__ h0, const float* __restrict__ c0,
                      int64_t state_dir_stride, const float* __restrict__ whh0, const float* __restrict__ whh1,
                      float* __restrict__ dz, float* __restrict__ hprev, int H, int T, int64_t n) {
    extern __shared__ float smem[];
    float* dzs = smem;                   // [4H][TS]
    float* dhr = dzs + 4 * H * TS_;      // [TS][H]
    float* dcs = dhr + TS_ * H;          // [TS][H]
    const int dir = blockIdx.y;
    const float* __restrict__ whh = dir ? whh1 : whh0;
    const int64_t site0 = (int64_t)blockIdx.x * TS_;
    const int tid = threadIdx.x, nthr = blockDim.x;
    for (int i = tid; i < TS_ * H; i += nthr) { dhr[i] = 0.f; dcs[i] = 0.f; }
    __syncthreads();
    for (int step = 0; step < T; ++step) {
        const int t = dir ? step : (T - 1 - step);
        const bool has_prev = dir ? (t < T - 1) : (t > 0);
        const int tp = dir ? t + 1 : t - 1;
        for (int j = tid; j < H; j += nthr) {
            for (int s = 0; s < TS_; ++s) {
                const int64_t site = site0 + s;
                float zi = 0.f, zf = 0.f, zg = 0.f, zo = 0.f;
                if (site < n) {
                    const int64_t rd = (site * T + t) * 2 + dir;
                    const float* gp = gates + rd * 4 * H + j;
                    const float ig = gp[0], fg = gp[H], gg = gp[2 * H], og = gp[3 * H];
                    const float c = cst[rd * H + j];
                    float cp, hp;
                    if (has_prev) {
                        cp = cst[((site * T + tp) * 2 + dir) * H + j];
                        hp = y[(site * T + tp) * (2 * (int64_t)H) + dir * H + j];
                    } else {
                        cp = c0[dir * state_dir_stride + site * H + j];
                        hp = h0[dir * state_dir_stride + site * H + j];
                    }
                    const float dh = dy[(site * T + t) * (2 * (int64_t)H) + dir * H + j] + dhr[s * H + j];
                    const float tc = tanhf(c);
                    const float dc = dcs[s * H + j] + dh * og * (1.f - tc * tc);
                    zi = dc * gg * ig * (1.f - ig);
                    zf = dc * cp * fg * (1.f - fg);
                    zg = dc * ig * (1.f - gg * gg);
                    zo = dh * tc * og * (1.f - og);
                    dcs[s * H + j] = dc * fg;
                    float* zp = dz + rd * 4 * H + j;
                    zp[0] = zi; zp[H] = zf; zp[2 * H] = zg; zp[3 * H] = zo;
                    hprev[(site * T + t) * (2 * (int64_t)H) + dir * H + j] = hp;
                }
                dzs[(0 * H + j) * TS_ + s] = zi;
                dzs[(1 * H + j) * TS_ + s] = zf;
                dzs[(2 * H + j) * TS_ + s] = zg;
                dzs[(3 * H + j) * TS_ + s] = zo;
            }
        }
        __syncthreads();
        for (int k = tid; k < H; k += nthr) {
            float acc[TS_];
#pragma unroll
            for (int s = 0; s < TS_; ++s) acc[s] = 0.f;
            for (int r = 0; r < 4 * H; ++r) {
                const float w = __ldg(whh + (int64_t)r * H + k);
#pragma unroll
                for (int s = 0; s < TS_; s += 4) {
                    const float4 d = *reinterpret_cast<const float4*>(dzs + r * TS_ + s);
                    acc[s] = fmaf(d.x, w, acc[s]);
                    acc[s + 1] = fmaf(d.y, w, acc[s + 1]);
                    acc[s + 2] = fmaf(d.z, w, acc[s + 2]);
                    acc[s + 3] = fmaf(d.w, w, acc[s + 3]);
                }
            }
#pragma unroll
            for (int s = 0; s < TS_; ++s) dhr[s * H + k] = acc[s];
        }
        __syncthreads();
    }
}

// C[m][n] (+)= sum_k A(m,k) B(k,n) (+ bias[n], ReLU) with arbitrary element strides, fp32 FMA.
// 64x64 tile, 16-deep k slices, 256 threads x 4x4 outputs.  blockIdx.z is the split-K index: with
// `partial` set, split z writes its sum over k in [z*kps, (z+1)*kps) to partial[z][M][N] and
// splitk_reduce_kernel adds the splits in order.
constexpr int GBM = 64, GBN = 64, GBK = 16;

__global__ void __launch_bounds__(256)
gemm_f32_kernel(int M, int N, int K, const float* __restrict__ A, int64_t sam, int64_t sak,
                const float* __restrict__ B, int64_t sbk, int64_t sbn, float* __restrict__ C, int64_t ldc,
                const float* __restrict__ bias, int relu, int beta, int kps, float* __restrict__ partial) {
    __shared__ float As[GBK][GBM + 4];
    __shared__ float Bs[GBK][GBN + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.x * GBM, n0 = blockIdx.y * GBN;
    const int kbeg = blockIdx.z * kps, kend = min(K, kbeg + kps);
    float acc[4][4] = {};
    for (int k0 = kbeg; k0 < kend; k0 += GBK) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = tid + i * 256;
            int mm, kk;
            if (sak == 1) { kk = idx & 15; mm = idx >> 4; } else { mm = idx & 63; kk = idx >> 6; }
            const int gm = m0 + mm, gk = k0 + kk;
            As[kk][mm] = (gm < M && gk < kend) ? A[(int64_t)gm * sam + (int64_t)gk * sak] : 0.f;
            int nn;
            if (sbn == 1) { nn = idx & 63; kk = idx >> 6; } else { kk = idx & 15; nn = idx >> 4; }
            const int gn = n0 + nn, gk2 = k0 + kk;
            Bs[kk][nn] = (gn < N && gk2 < kend) ? B[(int64_t)gk2 * sbk + (int64_t)gn * sbn] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GBK; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int gm = m0 + ty * 4 + i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gn = n0 + tx * 4 + j;
            if (gn >= N) continue;
            if (partial) {
                partial[((int64_t)blockIdx.z * M + gm) * N + gn] = acc[i][j];
            } else {
                float v = acc[i][j];
                float* c = C + (int64_t)gm * ldc + gn;
                if (beta) v += *c;
                if (bias) v += bias[gn];
                if (relu) v = fmaxf(v, 0.f);
                *c = v;
            }
        }
    }
}

__global__ void splitk_reduce_kernel(const float* __restrict__ partial, int splits, int M, int N,
                                     float* __restrict__ C, int64_t ldc, int beta) {
    const int64_t total = (int64_t)M * N;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        float v = 0.f;
        for (int z = 0; z < splits; ++z) v += partial[(int64_t)z * total + i];
        const int64_t m = i / N, nn = i - m * N;
        float* c = C + m * ldc + nn;
        *c = beta ? *c + v : v;
    }
}

// partial[z][c] = sum of x[r][c] over the rows of split z, in row order.
__global__ void colsum_partial_kernel(const float* __restrict__ x, int64_t ld, int64_t rows, int cols,
                                      int64_t rps, float* __restrict__ partial) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cols) return;
    const int64_t r0 = (int64_t)blockIdx.y * rps, r1 = min(rows, r0 + rps);
    float acc = 0.f;
    for (int64_t r = r0; r < r1; ++r) acc += x[r * ld + c];
    partial[(int64_t)blockIdx.y * cols + c] = acc;
}

// out[r][c] = g[r][c] * mask[r][c] (mask may be NULL), zeroed where act[r][c] <= 0 (act may be NULL),
// then ReLU if `relu`.  Dropout forward/backward, ReLU backward, and the head's relu(dropout(z1)).
__global__ void ew_kernel(float* __restrict__ out, int64_t ldo, const float* __restrict__ g, int64_t ldg,
                          const float* __restrict__ mask, int64_t ldm, const float* __restrict__ act, int64_t lda,
                          int relu, int64_t rows, int cols) {
    const int64_t total = rows * cols;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / cols, c = i - r * cols;
        float v = g[r * ldg + c];
        if (mask) v *= mask[r * ldm + c];
        if (act && !(act[r * lda + c] > 0.f)) v = 0.f;
        if (relu) v = fmaxf(v, 0.f);
        out[r * ldo + c] = v;
    }
}

// models.py:229-233: [h_fwd(T-1) | h_bwd(0)] of the last comb layer, times the first head dropout mask.
__global__ void pick_last_kernel(const float* __restrict__ y, int H, int T, int64_t n, const float* __restrict__ mask,
                                 float* __restrict__ out) {
    const int64_t total = n * 2 * H;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / (2 * H);
        const int k = (int)(i - r * 2 * H);
        const int t = k < H ? T - 1 : 0;
        float v = y[(r * T + t) * 2 * H + k];
        if (mask) v *= mask[i];
        out[i] = v;
    }
}

// Its backward: dY of the last comb layer is dlast (times the mask) at t = T-1 forward / t = 0 reverse, 0 elsewhere.
__global__ void scatter_last_kernel(const float* __restrict__ dlast, const float* __restrict__ mask, int H, int T,
                                    int64_t n, float* __restrict__ dy) {
    const int64_t total = n * T * 2 * H;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / (T * 2 * H);
        const int rem = (int)(i - r * T * 2 * H);
        const int t = rem / (2 * H), k = rem - t * 2 * H;
        float v = 0.f;
        if ((k < H && t == T - 1) || (k >= H && t == 0)) {
            v = dlast[r * 2 * H + k];
            if (mask) v *= mask[r * 2 * H + k];
        }
        dy[i] = v;
    }
}

// Embedding gradient: one CTA per code; each thread sums the rows r = tid, tid + 256, ... in order, then a
// fixed-shape tree over the 256 partial sums.
__global__ void __launch_bounds__(256)
embed_grad_kernel(const float* __restrict__ dx, int ldx, const int32_t* __restrict__ codes, int64_t rows, int E,
                  float* __restrict__ grad) {
    __shared__ float red[256];
    const int code = blockIdx.x;
    for (int e = 0; e < E; ++e) {
        float acc = 0.f;
        for (int64_t r = threadIdx.x; r < rows; r += 256)
            if (codes[r] == code) acc += dx[r * ldx + e];
        red[threadIdx.x] = acc;
        __syncthreads();
        for (int w = 128; w > 0; w >>= 1) {
            if ((int)threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
            __syncthreads();
        }
        if (threadIdx.x == 0) grad[code * E + e] = red[0];
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------
// Host side.

unsigned ew_grid(int64_t total) {
    int64_t b = (total + 255) / 256;
    return (unsigned)(b < 1 ? 1 : (b > 65535 * 8 ? 65535 * 8 : b));
}

int64_t splits_for(int64_t rows) {
    int64_t s = (rows + 2047) / 2048;
    return s < 1 ? 1 : (s > 64 ? 64 : s);
}

struct Stack { int layers, K0, H; };

// Sizes the training path derives from the configuration.
struct Shape {
    int T, S, H, C, kseq, E;
    bool seq, sig;
    Stack st[3];              // seq, signal, comb (layers == 0: absent)
    int n_params, n_masks;
};

Shape shape_of(const Model* m) {
    const dsp_config& c = m->cfg;
    Shape s;
    s.T = c.seq_len; s.S = c.signal_len; s.H = c.hidden_size; s.C = c.num_classes; s.kseq = m->kseq;
    s.E = c.is_base ? c.embedding_size : 0;
    s.seq = c.module != DSP_SIGNAL_BILSTM;
    s.sig = c.module != DSP_SEQ_BILSTM;
    s.st[0] = {s.seq ? c.num_layers2 : 0, m->kseq, m->nhid_seq};
    s.st[1] = {s.sig ? c.num_layers2 : 0, c.signal_len, m->nhid_signal};
    s.st[2] = {c.num_layers1, c.hidden_size, c.hidden_size};
    s.n_params = (s.seq ? 1 + 8 * c.num_layers2 + 2 : 0) + (s.sig ? 8 * c.num_layers2 + 2 : 0) + 8 * c.num_layers1 + 4;
    s.n_masks = 2 * (c.num_layers2 - 1) + (c.num_layers1 - 1) + 2;
    return s;
}

// Byte layout of a region: sections appended at 256-byte alignment.
struct Bump {
    char* base; size_t off = 0;
    explicit Bump(void* b) : base((char*)b) {}
    template <class X> X* take(int64_t count) {
        X* p = base ? (X*)(base + off) : nullptr;
        off += ((size_t)count * sizeof(X) + 255) & ~(size_t)255;
        return p;
    }
};

struct LayerAct {            // saved activations of one LSTM layer
    float* y; float* ym; float* gates; float* cst;
    float* wt[2]; float* bias[2];
};

// The arena: everything backward needs from one forward.  With base == nullptr only sizes are computed.
struct Arena {
    std::vector<LayerAct> layer[3];
    float* h0[3] = {}; float* c0[3] = {};
    float* xseq = nullptr; int32_t* codes = nullptr; float* sig = nullptr;
    float* comb_in = nullptr; float* in1 = nullptr; float* z1 = nullptr; float* a2 = nullptr;
    size_t bytes = 0;
    Arena(const Shape& s, int64_t n, void* base) {
        Bump b(base);
        const int64_t NT = n * s.T;
        for (int g = 0; g < 3; ++g) {
            const Stack& k = s.st[g];
            if (!k.layers) continue;
            h0[g] = b.take<float>((int64_t)k.layers * 2 * n * k.H);
            c0[g] = b.take<float>((int64_t)k.layers * 2 * n * k.H);
            for (int l = 0; l < k.layers; ++l) {
                const int K = l ? 2 * k.H : k.K0;
                LayerAct a;
                a.y = b.take<float>(NT * 2 * k.H);
                a.ym = (l + 1 < k.layers) ? b.take<float>(NT * 2 * k.H) : nullptr;
                a.gates = b.take<float>(NT * 2 * 4 * k.H);
                a.cst = b.take<float>(NT * 2 * k.H);
                for (int d = 0; d < 2; ++d) {
                    a.wt[d] = b.take<float>((int64_t)(ru(K, 4) + ru(k.H, 4)) * 4 * k.H);
                    a.bias[d] = b.take<float>(4 * k.H);
                }
                layer[g].push_back(a);
            }
        }
        if (s.seq) { xseq = b.take<float>(NT * s.kseq); codes = b.take<int32_t>(NT); }
        if (s.sig) sig = b.take<float>(NT * s.S);
        comb_in = b.take<float>(NT * s.H);
        in1 = b.take<float>(n * 2 * s.H);
        z1 = b.take<float>(n * s.H);
        a2 = b.take<float>(n * s.H);
        bytes = b.off;
    }
};

// Backward scratch.
struct Work {
    float* dy[2]; float* dz; float* hprev; float* dcomb; float* dfc; float* dxseq;
    float* dlast; float* da2; float* dz1; float* dbias; float* partial;
    int64_t partial_floats;
    size_t bytes;
    Work(const Shape& s, int64_t n, void* base) {
        Bump b(base);
        const int64_t NT = n * s.T;
        int64_t maxmn = 8 * (int64_t)s.H, hmax = s.H;
        for (int g = 0; g < 3; ++g) {
            const Stack& k = s.st[g];
            if (!k.layers) continue;
            if (k.H > hmax) hmax = k.H;
            for (int l = 0; l < k.layers; ++l) {
                const int64_t K = l ? 2 * k.H : k.K0;
                maxmn = std::max(maxmn, 4 * k.H * std::max(K, (int64_t)k.H));
            }
            if (g < 2) maxmn = std::max(maxmn, (int64_t)k.H * 2 * k.H);
        }
        maxmn = std::max(maxmn, (int64_t)s.H * 2 * s.H);
        dy[0] = b.take<float>(NT * 2 * hmax);
        dy[1] = b.take<float>(NT * 2 * hmax);
        dz = b.take<float>(NT * 8 * hmax);
        hprev = b.take<float>(NT * 2 * hmax);
        dcomb = b.take<float>(NT * s.H);
        dfc = b.take<float>(NT * hmax);
        dxseq = b.take<float>(NT * s.kseq);
        dlast = b.take<float>(n * 2 * s.H);
        da2 = b.take<float>(n * s.H);
        dz1 = b.take<float>(n * s.H);
        dbias = b.take<float>(8 * hmax);
        partial_floats = splits_for(NT) * maxmn;
        partial = b.take<float>(partial_floats);
        bytes = b.off;
    }
};

// Parameter (or gradient) pointers in state_dict order (models.py:131-161 creation order):
// embed, lstm_seq (8 per layer: weight_ih, weight_hh, bias_ih, bias_hh, then the same for _reverse), fc_seq,
// lstm_signal, fc_signal, lstm_comb, fc1, fc2.
template <class P>
struct Slots {
    P* embed = nullptr;
    std::vector<std::array<P*, 8>> lstm[3];
    P* fcw[2] = {}; P* fcb[2] = {};
    P* head[4] = {};             // fc1.weight, fc1.bias, fc2.weight, fc2.bias
    Slots(const Shape& s, P* list) {
        int i = 0;
        if (s.seq) embed = &list[i++];
        for (int g = 0; g < 3; ++g) {
            for (int l = 0; l < s.st[g].layers; ++l) {
                std::array<P*, 8> a;
                for (int q = 0; q < 8; ++q) a[q] = &list[i++];
                lstm[g].push_back(a);
            }
            if (g < 2 && s.st[g].layers) { fcw[g] = &list[i++]; fcb[g] = &list[i++]; }
        }
        for (int q = 0; q < 4; ++q) head[q] = &list[i++];
    }
};

// first dropout-mask slot of each stack's inter-layer masks (seq, signal, comb); the head's two come last
void mask_bases(const Model* m, int base[3]) {
    base[0] = 0;
    base[1] = m->cfg.num_layers2 - 1;
    base[2] = 2 * (m->cfg.num_layers2 - 1);
}

int launch_gemm(Model* m, int M, int N, int K, const float* A, int64_t sam, int64_t sak, const float* B, int64_t sbk,
                int64_t sbn, float* C, int64_t ldc, const float* bias, int relu, int beta, const Work* w, cudaStream_t st) {
    if (M == 0 || N == 0) return DSP_OK;
    int splits = 1, kps = K;
    if (w) {
        splits = (int)splits_for(K);
        kps = (int)((K + splits - 1) / splits);
        splits = (K + kps - 1) / kps;
        if (splits < 1) splits = 1;
    }
    float* partial = (w && splits > 1) ? w->partial : nullptr;
    if (partial && (int64_t)splits * M * N > w->partial_floats) {
        set_error("training GEMM %dx%d needs more split-K scratch than reserved", M, N);
        return DSP_ERR_INVALID;
    }
    dim3 grid((unsigned)((M + GBM - 1) / GBM), (unsigned)((N + GBN - 1) / GBN), (unsigned)splits);
    gemm_f32_kernel<<<grid, 256, 0, st>>>(M, N, K, A, sam, sak, B, sbk, sbn, C, ldc, bias, relu, beta, kps, partial);
    m->launches++;
    DSP_CUDA(cudaGetLastError());
    if (partial) {
        DSP_REQUIRE(!bias && !relu, DSP_ERR_INVALID, "split-K GEMM has no bias/ReLU epilogue");
        splitk_reduce_kernel<<<ew_grid((int64_t)M * N), 256, 0, st>>>(partial, splits, M, N, C, ldc, beta);
        m->launches++;
        DSP_CUDA(cudaGetLastError());
    }
    return DSP_OK;
}

// out[c] = sum over rows of x[r][c], fixed-order split over rows.
int launch_colsum(Model* m, const float* x, int64_t ld, int64_t rows, int cols, float* out, const Work& w, cudaStream_t st) {
    const int64_t splits0 = splits_for(rows), rps = (rows + splits0 - 1) / splits0;
    const int splits = (int)((rows + rps - 1) / rps);
    DSP_REQUIRE((int64_t)splits * cols <= w.partial_floats, DSP_ERR_INVALID, "bias gradient scratch too small");
    dim3 grid((unsigned)((cols + 255) / 256), (unsigned)splits);
    colsum_partial_kernel<<<grid, 256, 0, st>>>(x, ld, rows, cols, rps, w.partial);
    m->launches++;
    DSP_CUDA(cudaGetLastError());
    splitk_reduce_kernel<<<ew_grid(cols), 256, 0, st>>>(w.partial, splits, 1, cols, out, cols, 0);
    m->launches++;
    DSP_CUDA(cudaGetLastError());
    return DSP_OK;
}

int launch_ew(Model* m, float* out, int64_t ldo, const float* g, int64_t ldg, const float* mask, int64_t ldm,
              const float* act, int64_t lda, int relu, int64_t rows, int cols, cudaStream_t st) {
    if (rows * cols == 0) return DSP_OK;
    ew_kernel<<<ew_grid(rows * cols), 256, 0, st>>>(out, ldo, g, ldg, mask, ldm, act, lda, relu, rows, cols);
    m->launches++;
    DSP_CUDA(cudaGetLastError());
    return DSP_OK;
}

#define RC(x) do { int rc__ = (x); if (rc__) return rc__; } while (0)

}  // namespace

int train_shape(const Model* m, int32_t* n_params, int32_t* n_masks) {
    Shape s = shape_of(m);
    if (n_params) *n_params = s.n_params;
    if (n_masks) *n_masks = s.n_masks;
    return DSP_OK;
}

int64_t train_arena_bytes(const Model* m, int64_t n) { return (int64_t)Arena(shape_of(m), n, nullptr).bytes; }
int64_t train_workspace_bytes(const Model* m, int64_t n) { return (int64_t)Work(shape_of(m), n, nullptr).bytes; }

int train_forward(Model* m, const float* const* params, const float* kmer, const float* means, const float* stds,
                  const float* lens, const float* signals, const float* const* states6, uint64_t seed,
                  const float* const* masks, int64_t n, void* arena, float* logits, cudaStream_t st) {
    const Shape s = shape_of(m);
    Arena A(s, n, arena);
    Slots<const float* const> P(s, params);
    const int T = s.T, H = s.H;
    const int64_t NT = n * T;

    // initial states: copied from the caller or drawn (Philox, one stream per group); backward reads them here
    for (int g = 0; g < 3; ++g) {
        const Stack& k = s.st[g];
        if (!k.layers) continue;
        const int64_t cnt = (int64_t)k.layers * 2 * n * k.H;
        if (states6) {
            DSP_REQUIRE(states6[2 * g] && states6[2 * g + 1], DSP_ERR_INVALID, "dsp_train_forward: states[%d] is null", 2 * g);
            DSP_CUDA(cudaMemcpyAsync(A.h0[g], states6[2 * g], cnt * sizeof(float), cudaMemcpyDeviceToDevice, st));
            DSP_CUDA(cudaMemcpyAsync(A.c0[g], states6[2 * g + 1], cnt * sizeof(float), cudaMemcpyDeviceToDevice, st));
        } else {
            RC(philox_normal(m, A.h0[g], cnt, seed, 2 * g, st));
            RC(philox_normal(m, A.c0[g], cnt, seed, 2 * g + 1, st));
        }
    }
    // weights of every LSTM layer -> the forward kernel's layout, in the arena
    for (int g = 0; g < 3; ++g)
        for (int l = 0; l < s.st[g].layers; ++l) {
            const int K = l ? 2 * s.st[g].H : s.st[g].K0, Hh = s.st[g].H;
            for (int d = 0; d < 2; ++d) {
                const int64_t total = (int64_t)(ru(K, 4) + ru(Hh, 4)) * 4 * Hh;
                repack_lstm_kernel<<<ew_grid(total), 256, 0, st>>>(
                    *P.lstm[g][l][4 * d], *P.lstm[g][l][4 * d + 1], *P.lstm[g][l][4 * d + 2], *P.lstm[g][l][4 * d + 3],
                    K, Hh, A.layer[g][l].wt[d], A.layer[g][l].bias[d]);
                m->launches++;
                DSP_CUDA(cudaGetLastError());
            }
        }
    DSP_CUDA(cudaFuncSetAttribute(lstm_train_fwd_kernel<TS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));

    // one stack: layers in order, inter-layer dropout on every output but the last
    int mask_base[3];
    mask_bases(m, mask_base);
    auto run_stack = [&](int g, const float* x, int xs, int xt) -> const float* {
        const Stack& k = s.st[g];
        const int64_t sstride = n * k.H;
        for (int l = 0; l < k.layers; ++l) {
            const int K = l ? 2 * k.H : k.K0;
            LayerAct& a = A.layer[g][l];
            const size_t smem = sizeof(float) * TS * (size_t)(ru(K, 4) + 3 * ru(k.H, 4));
            if (smem > 227 * 1024) { set_error("training LSTM layer K=%d H=%d exceeds shared memory", K, k.H); return nullptr; }
            const int threads = k.H >= 256 ? 256 : ru(k.H, 32);
            lstm_train_fwd_kernel<TS><<<dim3((unsigned)((n + TS - 1) / TS), 2), threads, smem, st>>>(
                x, xs, xt, K, a.wt[0], a.wt[1], a.bias[0], a.bias[1], A.h0[g] + (int64_t)l * 2 * sstride,
                A.c0[g] + (int64_t)l * 2 * sstride, sstride, a.y, a.gates, a.cst, k.H, T, n);
            m->launches++;
            if (cudaGetLastError() != cudaSuccess) { set_error("lstm_train_fwd_kernel launch failed"); return nullptr; }
            x = a.y;
            const float* mk = (l + 1 < k.layers) ? masks[mask_base[g] + l] : nullptr;
            if (mk) {
                if (launch_ew(m, a.ym, 2 * k.H, a.y, 2 * k.H, mk, 2 * k.H, nullptr, 0, 0, NT, 2 * k.H, st)) return nullptr;
                x = a.ym;
            }
            xs = T * 2 * k.H; xt = 2 * k.H;
        }
        return x;
    };

    int comb_off = 0;
    if (s.seq) {
        assemble_seq_train_kernel<<<(unsigned)((NT + 255) / 256), 256, 0, st>>>(
            kmer, means, stds, lens, *P.embed, s.E, m->cfg.vocab_size, m->cfg.is_signallen, s.kseq, NT, A.xseq, A.codes);
        m->launches++;
        DSP_CUDA(cudaGetLastError());
        const float* y = run_stack(0, A.xseq, T * s.kseq, s.kseq);
        if (!y) return DSP_ERR_CUDA;
        const int hs = s.st[0].H;
        RC(launch_gemm(m, (int)NT, hs, 2 * hs, y, 2 * hs, 1, *P.fcw[0], 1, 2 * hs, A.comb_in, H, *P.fcb[0], 1, 0, nullptr, st));
        comb_off = hs;
    }
    if (s.sig) {
        DSP_CUDA(cudaMemcpyAsync(A.sig, signals, NT * s.S * sizeof(float), cudaMemcpyDeviceToDevice, st));
        const float* y = run_stack(1, A.sig, T * s.S, s.S);
        if (!y) return DSP_ERR_CUDA;
        const int hs = s.st[1].H;
        RC(launch_gemm(m, (int)NT, hs, 2 * hs, y, 2 * hs, 1, *P.fcw[1], 1, 2 * hs, A.comb_in + comb_off, H, *P.fcb[1], 1, 0,
                       nullptr, st));
    }
    const float* y = run_stack(2, A.comb_in, T * H, H);
    if (!y) return DSP_ERR_CUDA;
    // head: dropout -> fc1 -> dropout -> ReLU -> fc2 (models.py:229-238)
    const float* m1 = masks[s.n_masks - 2];
    const float* m2 = masks[s.n_masks - 1];
    pick_last_kernel<<<ew_grid(n * 2 * H), 256, 0, st>>>(y, H, T, n, m1, A.in1);
    m->launches++;
    DSP_CUDA(cudaGetLastError());
    RC(launch_gemm(m, (int)n, H, 2 * H, A.in1, 2 * H, 1, *P.head[0], 1, 2 * H, A.z1, H, *P.head[1], 0, 0, nullptr, st));
    RC(launch_ew(m, A.a2, H, A.z1, H, m2, H, nullptr, 0, 1, n, H, st));
    RC(launch_gemm(m, (int)n, s.C, H, A.a2, H, 1, *P.head[2], 1, H, logits, s.C, *P.head[3], 0, 0, nullptr, st));
    return DSP_OK;
}

int train_backward(Model* m, const float* const* params, const float* const* masks, const void* arena,
                   const float* dlogits, int64_t n, void* workspace, float* const* grads, cudaStream_t st) {
    const Shape s = shape_of(m);
    Arena A(s, n, const_cast<void*>(arena));
    Work W(s, n, workspace);
    Slots<const float* const> P(s, params);
    Slots<float* const> G(s, grads);
    const int T = s.T, H = s.H, C = s.C;
    const int64_t NT = n * T;
    const float* m1 = masks[s.n_masks - 2];
    const float* m2 = masks[s.n_masks - 1];

    // head (models.py:234-238)
    RC(launch_gemm(m, C, H, (int)n, dlogits, 1, C, A.a2, H, 1, *G.head[2], H, nullptr, 0, 0, &W, st));      // dW2
    RC(launch_colsum(m, dlogits, C, n, C, *G.head[3], W, st));                                               // db2
    RC(launch_gemm(m, (int)n, H, C, dlogits, C, 1, *P.head[2], H, 1, W.da2, H, nullptr, 0, 0, nullptr, st)); // da2
    RC(launch_ew(m, W.dz1, H, W.da2, H, m2, H, A.a2, H, 0, n, H, st));
    RC(launch_gemm(m, H, 2 * H, (int)n, W.dz1, 1, H, A.in1, 2 * H, 1, *G.head[0], 2 * H, nullptr, 0, 0, &W, st)); // dW1
    RC(launch_colsum(m, W.dz1, H, n, H, *G.head[1], W, st));                                                        // db1
    RC(launch_gemm(m, (int)n, 2 * H, H, W.dz1, H, 1, *P.head[0], 2 * H, 1, W.dlast, 2 * H, nullptr, 0, 0, nullptr, st));
    scatter_last_kernel<<<ew_grid(NT * 2 * H), 256, 0, st>>>(W.dlast, m1, H, T, n, W.dy[0]);
    m->launches++;
    DSP_CUDA(cudaGetLastError());

    DSP_CUDA(cudaFuncSetAttribute(lstm_train_bwd_kernel<TS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    int mask_base[3];
    mask_bases(m, mask_base);
    // one stack top-down; dY of its last layer is in W.dy[0]; dX of layer 0 goes to dx0 (ld = K0) unless dx0 is null
    auto back_stack = [&](int g, const float* x0, int ldx0, float* dx0) -> int {
        const Stack& k = s.st[g];
        const int64_t sstride = n * k.H;
        const int Hh = k.H;
        int cur = 0;
        for (int l = k.layers - 1; l >= 0; --l) {
            const LayerAct& a = A.layer[g][l];
            const int K = l ? 2 * Hh : k.K0;
            const float* x = l ? (A.layer[g][l - 1].ym && masks[mask_base[g] + l - 1] ? A.layer[g][l - 1].ym
                                                                                       : A.layer[g][l - 1].y)
                               : x0;
            const int ldx = l ? 2 * Hh : ldx0;
            const size_t smem = sizeof(float) * TS * (size_t)(4 * Hh + 2 * Hh);
            DSP_REQUIRE(smem <= 227 * 1024, DSP_ERR_INVALID, "training LSTM backward H=%d exceeds shared memory", Hh);
            const int threads = Hh >= 256 ? 256 : ru(Hh, 32);
            lstm_train_bwd_kernel<TS><<<dim3((unsigned)((n + TS - 1) / TS), 2), threads, smem, st>>>(
                W.dy[cur], a.gates, a.cst, a.y, A.h0[g] + (int64_t)l * 2 * sstride, A.c0[g] + (int64_t)l * 2 * sstride,
                sstride, *P.lstm[g][l][1], *P.lstm[g][l][5], W.dz, W.hprev, Hh, T, n);
            m->launches++;
            DSP_CUDA(cudaGetLastError());
            for (int d = 0; d < 2; ++d) {
                const float* dzd = W.dz + d * 4 * Hh;
                RC(launch_gemm(m, 4 * Hh, K, (int)NT, dzd, 1, 8 * Hh, x, ldx, 1, *G.lstm[g][l][4 * d], K, nullptr, 0, 0, &W, st));
                RC(launch_gemm(m, 4 * Hh, Hh, (int)NT, dzd, 1, 8 * Hh, W.hprev + d * Hh, 2 * Hh, 1, *G.lstm[g][l][4 * d + 1],
                               Hh, nullptr, 0, 0, &W, st));
            }
            RC(launch_colsum(m, W.dz, 8 * Hh, NT, 8 * Hh, W.dbias, W, st));
            for (int d = 0; d < 2; ++d) {
                DSP_CUDA(cudaMemcpyAsync(*G.lstm[g][l][4 * d + 2], W.dbias + d * 4 * Hh, 4 * Hh * sizeof(float),
                                         cudaMemcpyDeviceToDevice, st));
                DSP_CUDA(cudaMemcpyAsync(*G.lstm[g][l][4 * d + 3], W.dbias + d * 4 * Hh, 4 * Hh * sizeof(float),
                                         cudaMemcpyDeviceToDevice, st));
            }
            float* dx = l ? W.dy[cur ^ 1] : dx0;
            if (!dx) break;
            for (int d = 0; d < 2; ++d)
                RC(launch_gemm(m, (int)NT, K, 4 * Hh, W.dz + d * 4 * Hh, 8 * Hh, 1, *P.lstm[g][l][4 * d], K, 1, dx, K,
                               nullptr, 0, d, nullptr, st));
            if (l) {
                const float* mk = masks[mask_base[g] + l - 1];
                if (mk) RC(launch_ew(m, dx, K, dx, K, mk, K, nullptr, 0, 0, NT, K, st));
                cur ^= 1;
            }
        }
        return DSP_OK;
    };

    RC(back_stack(2, A.comb_in, H, W.dcomb));
    int comb_off = 0;
    for (int g = 0; g < 2; ++g) {
        if (!s.st[g].layers) continue;
        const int hs = s.st[g].H;
        const float* ytop = A.layer[g].back().y;
        float* dfc = W.dfc;
        // ReLU backward of the branch fc (models.py:199-201 / 215-217): comb_in holds relu(z)
        RC(launch_ew(m, dfc, hs, W.dcomb + comb_off, H, nullptr, 0, A.comb_in + comb_off, H, 0, NT, hs, st));
        RC(launch_gemm(m, hs, 2 * hs, (int)NT, dfc, 1, hs, ytop, 2 * hs, 1, *G.fcw[g], 2 * hs, nullptr, 0, 0, &W, st));
        RC(launch_colsum(m, dfc, hs, NT, hs, *G.fcb[g], W, st));
        RC(launch_gemm(m, (int)NT, 2 * hs, hs, dfc, hs, 1, *P.fcw[g], 2 * hs, 1, W.dy[0], 2 * hs, nullptr, 0, 0, nullptr, st));
        if (g == 0) {
            RC(back_stack(0, A.xseq, s.kseq, W.dxseq));
            if (s.E) {
                embed_grad_kernel<<<m->cfg.vocab_size, 256, 0, st>>>(W.dxseq, s.kseq, A.codes, NT, s.E, *G.embed);
                m->launches++;
                DSP_CUDA(cudaGetLastError());
            } else {
                DSP_CUDA(cudaMemsetAsync(*G.embed, 0, sizeof(float) * m->cfg.vocab_size * m->cfg.embedding_size, st));
            }
        } else {
            RC(back_stack(1, A.sig, s.S, nullptr));
        }
        comb_off += hs;
    }
    return DSP_OK;
}

}  // namespace dsp
