// Ranger (RAdam + Lookahead + gradient centralisation, the reference's utils/ranger2020.py) as one multi-tensor
// kernel: dsp_ranger_step updates every tensor of a parameter group in one launch (more than RG_MAXT tensors: one
// launch per RG_MAXT).
//
// Work items.  A centralised tensor (GC on and more than one dimension) is cut into its rows of row_len elements
// (size(0) rows); every other tensor into chunks of RG_TILE elements.  ONE WARP owns one item: it computes the row
// mean (gradient centralisation) with a fixed order -- each lane adds its elements in index order, then a butterfly
// over the 32 lanes, which leaves the same bits in every lane -- and updates the row in the same pass.  No atomics and
// no order that depends on scheduling: the same inputs give the same bits, on every call and every rank.
//
// Traffic.  A row of up to RG_TILE elements is held in registers: p, g, exp_avg and exp_avg_sq are read once and
// written once (g only when it is centralised in place), slow_buffer is read and written on Lookahead steps only.
// Longer rows read g a second time for the mean, and with gc_loc = 0 a centralised row computes the update twice
// (once for the mean of G, once to store it); both second reads hit L2.
//
// Arithmetic is fp32 in the published operation order; the scalars are rounded to float as torch rounds a Python
// number it applies to a float32 tensor.
#include "common.cuh"
#include <algorithm>
#include <cmath>

namespace dsp {
namespace {

constexpr int RG_MAXT = 56;                     // tensors per launch: the list stays in the 4 KB of kernel parameters
constexpr int RG_WARPS = 8;                     // warps (= work items) per CTA
constexpr int RG_EPT = 16;                      // elements per lane of one tile
constexpr int RG_TILE = 32 * RG_EPT;            // 512: the longest row both_bilstm has

struct RgList {
    float* p[RG_MAXT];
    float* g[RG_MAXT];
    float* m[RG_MAXT];
    float* v[RG_MAXT];
    float* slow[RG_MAXT];
    int64_t numel[RG_MAXT];
    int64_t item_len[RG_MAXT];                  // row_len of a centralised tensor, else RG_TILE
    int64_t item_off[RG_MAXT + 1];              // first work item of each tensor; item_off[count] = items of the launch
    float scale[RG_MAXT];                       // -step_size * lr
    uint8_t flags[RG_MAXT];                     // DSP_RANGER_*
    int count;
};
static_assert(sizeof(RgList) <= 4000, "the tensor list must fit the classic 4 KB of kernel parameters");

struct RgHyper {
    float beta1, beta2, c1, c2, eps, wd, alpha;  // c1 = float(1 - beta1), c2 = float(1 - beta2)
};

__device__ __forceinline__ int rg_find(const int64_t* off, int count, int64_t j) {
    int lo = 0, hi = count - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= j) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__device__ __forceinline__ float warp_sum(float x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = __fadd_rn(x, __shfl_xor_sync(0xffffffffu, x, o));
    return x;
}

// The moment updates and the search direction G of one element, before a gc_loc = 0 centralisation:
//   exp_avg_sq.mul_(beta2).addcmul_(g, g, value=1-beta2); exp_avg.mul_(beta1).add_(g, alpha=1-beta1)
//   G = exp_avg / (exp_avg_sq.sqrt() + eps) if rectified else exp_avg;  G.add_(p, alpha=weight_decay)
// Un-rectified, G IS exp_avg, so the weight decay lands in the stored moment as well.
__device__ __forceinline__ float rg_direction(float g, float p, float& m, float& v, bool rect, const RgHyper& h) {
    v = __fmul_rn(v, h.beta2) + h.c2 * g * g;
    m = __fmul_rn(m, h.beta1) + h.c1 * g;
    float G = rect ? __fdiv_rn(m, __fadd_rn(__fsqrt_rn(v), h.eps)) : m;
    if (h.wd != 0.f) G = G + h.wd * p;
    if (!rect) m = G;
    return G;
}

template <bool GC_LOC>
__global__ void __launch_bounds__(RG_WARPS * 32) ranger_kernel(const __grid_constant__ RgList l, const RgHyper h) {
    const int lane = threadIdx.x & 31;
    const int64_t item = (int64_t)blockIdx.x * RG_WARPS + (threadIdx.x >> 5);
    if (item >= l.item_off[l.count]) return;                 // whole warps leave together
    const int t = rg_find(l.item_off, l.count, item);
    const int64_t lo = (item - l.item_off[t]) * l.item_len[t];
    const int64_t len = min(l.item_len[t], l.numel[t] - lo);
    float* __restrict__ P = l.p[t] + lo;
    float* __restrict__ Gr = l.g[t] + lo;
    float* __restrict__ M = l.m[t] + lo;
    float* __restrict__ V = l.v[t] + lo;
    float* __restrict__ S = l.slow[t] + lo;
    const unsigned f = l.flags[t];
    const bool centre = f & DSP_RANGER_CENTRALIZE, rect = f & DSP_RANGER_RECTIFY, look = f & DSP_RANGER_LOOKAHEAD;
    const bool resident = len <= RG_TILE;
    const float scale = l.scale[t];

    float rg[RG_EPT];                                        // the gradient tile, kept from the mean to the update
    float mean = 0.f;
    if (centre) {                                            // the row mean of g (gc_loc) or of G (gc_loc = 0)
        float acc = 0.f;
        for (int64_t b = 0; b < len; b += RG_TILE) {
#pragma unroll
            for (int j = 0; j < RG_EPT; ++j) {
                const int64_t i = b + j * 32 + lane;
                if (i < len) {
                    const float g = Gr[i];
                    if (GC_LOC) {
                        rg[j] = g;
                        acc = __fadd_rn(acc, g);
                    } else {
                        float m = M[i], v = V[i];
                        rg[j] = g;
                        acc = __fadd_rn(acc, rg_direction(g, P[i], m, v, rect, h));
                    }
                }
            }
        }
        // as torch's mean kernel: the sum scaled by 1/n
        mean = __fmul_rn(warp_sum(acc), 1.0f / (float)len);
    }

    for (int64_t b = 0; b < len; b += RG_TILE) {
        float rp[RG_EPT], rm[RG_EPT], rv[RG_EPT], rs[RG_EPT];
#pragma unroll
        for (int j = 0; j < RG_EPT; ++j) {                   // every load of the tile before the first store
            const int64_t i = b + j * 32 + lane;
            if (i < len) {
                if (!(centre && resident)) rg[j] = Gr[i];
                rp[j] = P[i]; rm[j] = M[i]; rv[j] = V[i];
                if (look) rs[j] = S[i];
            }
        }
#pragma unroll
        for (int j = 0; j < RG_EPT; ++j) {
            const int64_t i = b + j * 32 + lane;
            if (i < len) {
                float g = rg[j], m = rm[j], v = rv[j];
                if (GC_LOC && centre) {                      // grad.add_(-mean): p.grad itself is centralised
                    g = __fsub_rn(g, mean);
                    Gr[i] = g;
                }
                float G = rg_direction(g, rp[j], m, v, rect, h);
                if (!GC_LOC && centre) {                     // G.add_(-mean(G)); un-rectified that is exp_avg
                    G = __fsub_rn(G, mean);
                    if (!rect) m = G;
                }
                float p = rp[j] + scale * G;                 // p.add_(G, alpha=-step_size * lr)
                if (look) {                                  // slow.add_(p - slow, alpha=alpha); p.copy_(slow)
                    const float s = rs[j] + h.alpha * __fsub_rn(p, rs[j]);
                    S[i] = s;
                    p = s;
                }
                P[i] = p; M[i] = m; V[i] = v;
            }
        }
    }
}

}  // namespace
}  // namespace dsp

using namespace dsp;

extern "C" int dsp_ranger_step(int32_t n_tensors, float* const* params, float* const* grads, float* const* exp_avg,
                               float* const* exp_avg_sq, float* const* slow_buffer, const int64_t* numel,
                               const int64_t* row_len, const float* neg_step_lr, const int32_t* flags, double beta1,
                               double beta2, double eps, double weight_decay, double alpha, int32_t gc_loc, void* stream) {
    DSP_REQUIRE(n_tensors >= 0, DSP_ERR_INVALID, "dsp_ranger_step: n_tensors=%d", (int)n_tensors);
    DSP_REQUIRE(n_tensors == 0 || (params && grads && exp_avg && exp_avg_sq && slow_buffer && numel && row_len && neg_step_lr && flags),
                DSP_ERR_INVALID, "dsp_ranger_step: null pointer list");
    DSP_REQUIRE(gc_loc == 0 || gc_loc == 1, DSP_ERR_INVALID, "dsp_ranger_step: gc_loc=%d", (int)gc_loc);
    const int32_t known = DSP_RANGER_RECTIFY | DSP_RANGER_LOOKAHEAD | DSP_RANGER_CENTRALIZE;
    for (int32_t i = 0; i < n_tensors; ++i) {
        DSP_REQUIRE(numel[i] >= 0, DSP_ERR_INVALID, "dsp_ranger_step: numel[%d]=%lld is negative", (int)i, (long long)numel[i]);
        DSP_REQUIRE(row_len[i] >= 1 && numel[i] % row_len[i] == 0, DSP_ERR_INVALID,
                    "dsp_ranger_step: row_len[%d]=%lld does not divide numel %lld", (int)i, (long long)row_len[i],
                    (long long)numel[i]);
        DSP_REQUIRE((flags[i] & ~known) == 0, DSP_ERR_INVALID, "dsp_ranger_step: flags[%d]=%d", (int)i, (int)flags[i]);
        DSP_REQUIRE(numel[i] == 0 || (params[i] && grads[i] && exp_avg[i] && exp_avg_sq[i] && slow_buffer[i]), DSP_ERR_INVALID,
                    "dsp_ranger_step: tensor %d has a null pointer", (int)i);
    }
    const RgHyper h{(float)beta1, (float)beta2, (float)(1.0 - beta1), (float)(1.0 - beta2), (float)eps, (float)weight_decay,
                    (float)alpha};
    cudaStream_t st = (cudaStream_t)stream;
    for (int32_t i0 = 0; i0 < n_tensors; i0 += RG_MAXT) {
        RgList l{};
        l.count = std::min<int32_t>(RG_MAXT, n_tensors - i0);
        int64_t items = 0;
        for (int k = 0; k < l.count; ++k) {
            const int i = i0 + k;
            l.p[k] = params[i]; l.g[k] = grads[i]; l.m[k] = exp_avg[i]; l.v[k] = exp_avg_sq[i]; l.slow[k] = slow_buffer[i];
            l.numel[k] = numel[i];
            l.item_len[k] = (flags[i] & DSP_RANGER_CENTRALIZE) ? row_len[i] : RG_TILE;
            l.scale[k] = neg_step_lr[i];
            l.flags[k] = (uint8_t)flags[i];
            l.item_off[k] = items;
            items += (numel[i] + l.item_len[k] - 1) / l.item_len[k];
        }
        l.item_off[l.count] = items;
        if (items == 0) continue;
        const int64_t blocks = (items + RG_WARPS - 1) / RG_WARPS;
        DSP_REQUIRE(blocks <= 0x7fffffff, DSP_ERR_INVALID, "dsp_ranger_step: %lld work items", (long long)items);
        if (gc_loc) ranger_kernel<true><<<(unsigned)blocks, RG_WARPS * 32, 0, st>>>(l, h);
        else ranger_kernel<false><<<(unsigned)blocks, RG_WARPS * 32, 0, st>>>(l, h);
        DSP_CUDA(cudaGetLastError());
    }
    return DSP_OK;
}
