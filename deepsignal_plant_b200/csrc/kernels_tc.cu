// tcgen05 / TMEM path of the ModelBiLSTM forward (DSP_PRECISION_FP16).
//
// Arithmetic: FP16 MMA operands (weights, layer inputs, h_{t-1}), FP32 accumulation in TMEM,
// FP32 bias, FP32 cell state and gate math.  Reference semantics: deepsignal_plant/models.py
// :178-240 and torch nn.LSTM (gate order i,f,g,o; reverse direction walks t = T-1..0).
//
// Data layout.  A site tile is 128 sites (= the 128 TMEM lanes of one SM).  Every MMA operand
// lives in HBM as "slabs" (rows x 64 fp16, 128-byte swizzled, see tc_prims.cuh) so that one
// linear cp.async.bulk brings it to shared memory ready for tcgen05.mma:
//   activations  [tile][t][slab][128 rows x 128 B]      (x_t of a layer = slabs of one (tile,t))
//   weights      [dir][cta rank][stream order][64 rows x 128 B]; a chunk = 128 gate columns =
//                32 hidden units x {i,f,g,o}; column n of a chunk = unit pair (n >> 3), gate
//                (n >> 1) & 3, unit parity n & 1 (adjacent columns = the same gate of two
//                adjacent units, so the epilogue works on packed fp32 pairs); CTA rank r of a
//                pair holds columns [64 r, 64 r + 64).
//
// A CTA PAIR (cluster of 2, tcgen05 cta_group::2, M = 256) owns two site tiles of one
// direction for all T steps; see layer_kernel.  Per step and chunk
//     acc[256 x 128] = x_t * W_ih_chunk^T      (A from shared memory)
//                    + h_{t-1} * W_hh_chunk^T  (A from TMEM)
// into one of two TMEM accumulators; the epilogue warps (thread = site) read their accumulator
// row, apply the gate non-linearities, update the cell state they keep in registers for all
// T steps, and write h_t as packed FP16 straight into the TMEM A operand of the next step and
// as a slab image to HBM for the next layer.  h and c never leave the SM between steps; gate
// pre-activations never touch HBM.
#include "tc.cuh"
#include "tc_prims.cuh"
#include <vector>
#include <cstring>
#include <cstdlib>

namespace dsp {

using namespace tc;

namespace {

constexpr int TILE = 128;
constexpr int SLAB_BYTES = TILE * SLAB_ROW_BYTES;   // 16 KB: one A-operand slab (128 site rows x 64 fp16)
constexpr int HSLAB_BYTES = SLAB_BYTES / 2;         // 8 KB: one CTA's half (64 weight rows) of a B slab
constexpr int EPI_WARPS = 16;                        // 4 per scheduler: enough independent work to keep the MUFU pipe busy
constexpr int NTHREADS = 128 + EPI_WARPS * 32;      // warps 0-3: producers / MMA issuer / TMEM; 4-19: epilogue
constexpr int CPT = 128 / (EPI_WARPS / 4);          // accumulator columns per epilogue thread per chunk (32)
constexpr int UPT = CPT / 4;                        // hidden units per epilogue thread per chunk (8)
constexpr float LOG2E = 1.4426950408889634f;
constexpr uint16_t PAIR_MASK = 3;                   // both CTAs of the pair

// Which of the five exponentials of an LSTM cell update are evaluated on the FMA pipe (degree-5
// polynomial, ~2e-7 relative error, same class as ex2.approx) instead of the 16-lane MUFU pipe:
// bit0 tanh(g), bit1 tanh(c), bit2 sigmoid(i), bit3 sigmoid(f), bit4 sigmoid(o).  With 16
// epilogue warps the MUFU pipe keeps up with the tensor pipe, and the whole step is bound by the
// 1 kW power cap, where one MUFU op costs less than the ~7 FMA-pipe instructions that replace
// it (measured, profiles/r01_run8_epilogue_variants.log): default 0.
#ifndef DSP_POLY_MASK
#define DSP_POLY_MASK 0
#endif
// The two branch layers (hidden 128, K = 16 + 128) are the exception: their MMAs are tiny, the SM runs
// far below the power cap and the MUFU pipe is what bounds them, so they get their own mask.
#ifndef DSP_POLY_MASK_BRANCH
#define DSP_POLY_MASK_BRANCH 3
#endif
// One reciprocal instead of two in the cell update (see lstm_cell2): fewer MUFU ops and, measured,
// ~2 % more sites/s at the power cap (profiles/r01_run12_epilogue_variants2.log).  0 = separate form.
// lstm_comb layer 0 (K = 256 + 256) sits between the two regimes.
#ifndef DSP_POLY_MASK_L0
#define DSP_POLY_MASK_L0 DSP_POLY_MASK
#endif
// Load the whole 32-column accumulator slice before the gate math in the hidden-256 layers too (frees
// the accumulator earlier, costs registers): measured 2 % slower (profiles/r01_run25_pw32_all_layers.log).
#ifndef DSP_PW32_ALL
#define DSP_PW32_ALL 0
#endif
#ifndef DSP_DIR_INTERLEAVE
#define DSP_DIR_INTERLEAVE 1
#endif
#ifndef DSP_MERGE_RCP
#define DSP_MERGE_RCP 1
#endif
// How the five non-linearities of a cell update are evaluated:
//   2 (default) all through MUFU tanh.approx.f32, sigmoid(z) = 0.5 + 0.5 tanh(0.5 z) with the 0.5 folded into the packed
//     weights: 5 MUFU ops and 3 packed FMA-pipe ops per unit-step;
//   0 every one as 2^x + reciprocal (ex2.approx / rcp.approx, ~1e-7 relative error): 7 MUFU and ~9 packed ops
//     (the DSP_POLY_MASK* / DSP_MERGE_RCP switches above only matter here);
//   1 sigmoid(o) and tanh(c') through tanh.approx, the rest as in 0 (the approximation enters h only, never c).
// Measured on 3 x 102 400 sites against the fp32 reference (profiles/r02_run17_tanh_approx_variants.log): label flips
// 1/0/0 (0), 2/0/0 (1), 4/0/0 (2) -- all inside the >= 99.99 % bar -- max |dprob| 5.5e-6 ... 7.0e-6 in all three, and
// 8.70 M / 8.95 M / 9.28 M sites/s: at the power cap the step follows energy per site, and 2 does a third of the
// epilogue arithmetic.  Build with -DDSP_TANH_APPROX=0 for the 1e-7 epilogue.
#ifndef DSP_TANH_APPROX
#define DSP_TANH_APPROX 2
#endif

struct LayerParams {
    const uint8_t* x_img;      // [tiles][T][KSX] slabs
    const uint8_t* w_img;      // [dir][cta rank][stream order] half slabs
    const float* bias;         // [dir][NCH*128] in chunk column order (LSTM: pre-scaled like the weights)
    const float* h0;           // [dir][n][H] fp32 (LSTM only); null: draw N(0,1) in-kernel (Philox)
    const float* c0;
    uint64_t seed;             // Philox key
    uint32_t rng_call;         // Philox counter word 3 (chunk / call id)
    uint32_t rng_slot;         // state slot id of this layer ((group*8 + layer) * 2), dir is added in-kernel
    int64_t site_base;         // global index of this chunk's first site
    int64_t state_dir_stride;
    uint8_t* y_img;            // output image: [tiles][T][y_slabs] slabs
    float* hfinal;             // [tiles*128][2H] fp32, last step of each direction (or null)
    int64_t n;
    int T;
    int xk16;                  // K16 steps of the x part (= KSX*4 unless the input is narrow)
    int y_slabs;
    int y_col_off;             // FC: first output column
    int write_y;               // 1: every step at (tile, t); 2: only the last step of the direction, at (tile, 0)
    // MODE_HEAD only
    const float* w2t;          // fc2 weight, [hidden][C]
    const float* b2;
    float* logits;
    float* probs;
    int32_t* labels;
    int num_classes;
};

enum { MODE_LSTM = 0, MODE_FC = 1, MODE_HEAD = 2 };
constexpr int HEAD_MAX_CLASSES = 8;
template <int KSX, int H, int MODE, int NOUT> struct LayerCfg {
    static constexpr int NCH = MODE != MODE_LSTM ? NOUT / 128 : H / 32;   // 128-column chunks per step
    // weight ring: NST stages of STG half slabs (one mbarrier pair per stage)
    static constexpr int STG = KSX >= 8 ? 2 : 4;
    static constexpr int NST = KSX >= 8 ? (MODE == 2 ? 4 : 5) : (MODE == 1 ? 2 : 4);
    // x_t buffers: the per-timestep dense layers are HBM-bound streams of x_t, so where shared memory allows
    // they double-buffer it (load of step t+1 overlaps the MMAs and stores of step t)
    static constexpr int XB = (MODE == 1 && KSX <= 4) ? 2 : 1;
    // dynamic shared memory, as offsets from its 1 KB-aligned base: XB x KSX x_t slabs at 0, the ring, the biases
    static constexpr size_t W = (size_t)KSX * XB * SLAB_BYTES;
    static constexpr size_t BIAS = W + (size_t)NST * STG * HSLAB_BYTES;
    static constexpr size_t BYTES = BIAS + (size_t)NCH * 128 * sizeof(float) + 1024;     // + the alignment slack
};

// Philox4x32-10 (Salmon et al., SC'11) + Box-Muller: four N(0,1) values per counter.  Used to
// draw the initial LSTM states in-kernel (the reference draws torch.randn per call,
// models.py:169-176), keyed by (seed; site, state slot, call) so no state ever crosses HBM.
__device__ __forceinline__ float4 philox_normal4(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    // uniforms in (0,1]: (x + 1) * 2^-32 never returns 0, so the log is finite
    const float u0 = ((float)c0 + 1.0f) * 2.3283064365386963e-10f, u1 = (float)c1 * 2.3283064365386963e-10f;
    const float u2 = ((float)c2 + 1.0f) * 2.3283064365386963e-10f, u3 = (float)c3 * 2.3283064365386963e-10f;
    const float r0 = sqrtf(-2.0f * __logf(u0)), r1 = sqrtf(-2.0f * __logf(u2));
    float s0, cs0, s1, cs1;
    __sincosf(6.283185307179586f * u1, &s0, &cs0);
    __sincosf(6.283185307179586f * u3, &s1, &cs1);
    return make_float4(r0 * cs0, r0 * s0, r1 * cs1, r1 * s1);
}

// ---- gate math on pairs of hidden units ---------------------------------------------------------
// 2^x for two values.  POLY: round-to-nearest split x = n + f, f in [-0.5, 0.5], degree-5
// polynomial for 2^f on the FMA pipe (packed FFMA2), n added into the exponent field;
// otherwise MUFU ex2.approx.  HI_CLAMP bounds the result (callers divide by 1 + result).
template <bool POLY, bool HI_CLAMP>
__device__ __forceinline__ float2 exp2_pair(float2 x) {
    if constexpr (POLY) {
        x.x = fmaxf(fminf(x.x, 40.f), -126.f);
        x.y = fmaxf(fminf(x.y, 40.f), -126.f);
        const float MG = 12582912.f;                      // 1.5 * 2^23: x + MG holds round(x) in its low mantissa bits
        const float2 t = add2(x, make_float2(MG, MG));
        const float2 r = add2(t, make_float2(-MG, -MG));
        const float2 f = fma2(r, make_float2(-1.f, -1.f), x);
        float2 q = fma2(make_float2(0.0013390863f, 0.0013390863f), f, make_float2(0.009676032f, 0.009676032f));
        q = fma2(q, f, make_float2(0.05550357f, 0.05550357f));
        q = fma2(q, f, make_float2(0.24022107f, 0.24022107f));
        q = fma2(q, f, make_float2(0.6931472f, 0.6931472f));
        q = fma2(q, f, make_float2(1.0000001f, 1.0000001f));
        q.x = __int_as_float(__float_as_int(q.x) + (__float_as_int(t.x) << 23));
        q.y = __int_as_float(__float_as_int(q.y) + (__float_as_int(t.y) << 23));
        return q;
    } else {
        if constexpr (HI_CLAMP) { x.x = fminf(x.x, 40.f); x.y = fminf(x.y, 40.f); }   // (1 + 2^40)^3 stays finite
        return make_float2(ex2_approx(x.x), ex2_approx(x.y));
    }
}

__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// scale folded into the packed weights and biases of gate g (0 i, 1 f, 2 g, 3 o)
__host__ __device__ inline float gate_scale(int g) {
#if DSP_TANH_APPROX == 2
    return g == 2 ? 1.f : 0.5f;                      // sigmoid(z) = 0.5 + 0.5 tanh(0.5 z)
#elif DSP_TANH_APPROX == 1
    return g == 2 ? -2.f * 1.4426950408889634f : (g == 3 ? 0.5f : -1.4426950408889634f);
#else
    return g == 2 ? -2.f * 1.4426950408889634f : -1.4426950408889634f;
#endif
}

// One LSTM cell update for two hidden units (torch nn.LSTM: c' = s(f) c + s(i) tanh(g),
// h = s(o) tanh(c')).  The inputs are the gate pre-activations already multiplied by
// -log2(e) (i, f, o) and -2 log2(e) (g) -- the factors are folded into the packed weights and
// biases -- so sigmoid(z) = 1 / (1 + 2^a) and tanh(z) = (1 - 2^a) / (1 + 2^a).
template <int PM>
__device__ __forceinline__ void lstm_cell2(float2 ai, float2 af, float2 ag, float2 ao, float2& c, float2& h) {
    const float2 ONE = make_float2(1.f, 1.f), NEG1 = make_float2(-1.f, -1.f);
#ifdef DSP_EPI_STUB   // measurement build only: no transcendental work, just enough arithmetic to keep every input live
    c = fma2(af, make_float2(1e-3f, 1e-3f), c);
    h = fma2(add2(ai, add2(ag, ao)), make_float2(1e-2f, 1e-2f), mul2(c, make_float2(1e-3f, 1e-3f)));
    return;
#endif
#if DSP_TANH_APPROX == 2
    {
        const float2 HALF = make_float2(0.5f, 0.5f);
        const float2 si = fma2(make_float2(tanh_approx(ai.x), tanh_approx(ai.y)), HALF, HALF);
        const float2 sf = fma2(make_float2(tanh_approx(af.x), tanh_approx(af.y)), HALF, HALF);
        const float2 so = fma2(make_float2(tanh_approx(ao.x), tanh_approx(ao.y)), HALF, HALF);
        const float2 tg = make_float2(tanh_approx(ag.x), tanh_approx(ag.y));
        c = fma2(sf, c, mul2(si, tg));
        h = mul2(so, make_float2(tanh_approx(c.x), tanh_approx(c.y)));
        return;
    }
#endif
#if DSP_MERGE_RCP
    constexpr bool CLAMP_IF = true;
#else
    constexpr bool CLAMP_IF = false;
#endif
    const float2 ei = exp2_pair<((PM >> 2) & 1) != 0, CLAMP_IF>(ai);
    const float2 ef = exp2_pair<((PM >> 3) & 1) != 0, CLAMP_IF>(af);
    const float2 eg = exp2_pair<(PM & 1) != 0, true>(ag);
    const float2 eo = exp2_pair<((PM >> 4) & 1) != 0, false>(ao);
#if DSP_MERGE_RCP
    // c' = [c (1+ei)(1+eg) + (1-eg)(1+ef)] / [(1+ef)(1+ei)(1+eg)]: one reciprocal instead of two
    // (needs bounded ei, ef: callers of this variant clamp them through HI_CLAMP below)
    const float2 F = add2(ef, ONE);
    const float2 AG = mul2(add2(ei, ONE), add2(eg, ONE));
    const float2 num = fma2(c, AG, mul2(fma2(eg, NEG1, ONE), F));
    const float2 den = mul2(F, AG);
    const float2 cn = mul2(num, make_float2(rcp_approx(den.x), rcp_approx(den.y)));
#else
    const float2 F = add2(ef, ONE);
    const float2 sf = make_float2(rcp_approx(F.x), rcp_approx(F.y));
    const float2 AG = mul2(add2(ei, ONE), add2(eg, ONE));
    const float2 rg = make_float2(rcp_approx(AG.x), rcp_approx(AG.y));
    const float2 ig = mul2(fma2(eg, NEG1, ONE), rg);                       // sigmoid(i) * tanh(g)
    const float2 cn = fma2(sf, c, ig);
#endif
    c = cn;
#if DSP_TANH_APPROX == 1
    {
        const float2 HALF = make_float2(0.5f, 0.5f);
        const float2 so = fma2(make_float2(tanh_approx(ao.x), tanh_approx(ao.y)), HALF, HALF);
        h = mul2(so, make_float2(tanh_approx(cn.x), tanh_approx(cn.y)));
        return;
    }
#endif
    const float2 ec = exp2_pair<((PM >> 1) & 1) != 0, true>(mul2(cn, make_float2(-2.f * LOG2E, -2.f * LOG2E)));
    const float2 D = mul2(add2(eo, ONE), add2(ec, ONE));
    const float2 rd = make_float2(rcp_approx(D.x), rcp_approx(D.y));
    h = mul2(fma2(ec, NEG1, ONE), rd);                                     // sigmoid(o) * tanh(c')
}

// ---------------------------------------------------------------------------------------------
// KSX: x slabs per step; H: hidden size of the layer (LSTM); MODE: what the epilogue does --
//   MODE_LSTM  recurrent layer (A = [x_t | h_{t-1}], gate math, cell update)
//   MODE_FC    dense + ReLU per timestep, NOUT output columns, written as a slab image
//   MODE_HEAD  fc1 + ReLU + fc2 + softmax (+argmax) on [h_fwd(T-1) | h_bwd(0)] (models.py:229-240)
//
// The kernel runs as CTA pairs (thread-block clusters of 2 on one TPC, tcgen05 cta_group::2):
// the two CTAs own two different site tiles of the same direction and execute every MMA
// together as M = 256.  Each CTA stages only HALF of every weight slab (64 of the 128 gate
// columns of a chunk), so the shared-memory fill rate per SM that bounds a single-CTA M = 128
// formulation (one full weight pass per tile and timestep) is halved.  The leader CTA (rank 0)
// issues all MMAs; completion is multicast to both CTAs' barriers; the peer CTA forwards its
// "data landed" and "accumulator drained" events to the leader's barriers.
//
// Warp roles (both CTAs unless noted):
//   warp 0     weight producer: streams this CTA's half slabs through a ring (cp.async.bulk)
//   warp 1     leader: MMA issuer / peer: relay of its full-barriers to the leader
//   warp 2     x_t slab producer (own tile)
//   warp 3     TMEM allocation
//   warps 4-19 epilogue, thread = (site row, 32-column slice of the chunk)
// Per step and chunk pair (c, c+1) the issue order is X(c) X(c+1) H(c) H(c+1), X = x_t part
// from shared memory into accumulator c&1, H = h_{t-1} part from TMEM, so that at a step
// boundary two x parts cover the tail of the previous step's gate math.
template <int KSX, int H, int MODE, int NOUT>
__global__ void __launch_bounds__(NTHREADS, 1)
layer_kernel(const LayerParams p) {
    constexpr bool IS_FC = MODE != MODE_LSTM;              // no recurrence: x part only
    using Cfg = LayerCfg<KSX, H, MODE, NOUT>;
    constexpr int STG = Cfg::STG, NST = Cfg::NST, XB = Cfg::XB;
    constexpr int NXS = KSX * XB;                          // x slabs resident in shared memory
    constexpr int NCH = Cfg::NCH;
    constexpr int KSH = IS_FC ? 0 : H / 64;                // h slabs (K of the recurrent part)
    constexpr int KS = KSX + KSH;
    constexpr int W_STEP = NCH * KS;                       // half slabs streamed per step
    constexpr int NBIAS = NCH * 128;
    constexpr uint32_t IDESC = make_idesc_f16(256, 128);
    static_assert(W_STEP % STG == 0, "a step must be a whole number of ring stages");
    static_assert(IS_FC || NCH % 2 == 0, "chunks are issued in pairs");
    static_assert(EPI_WARPS == 16 && CPT == 32 && UPT == 8, "the epilogue code below is written for 32-column slices");

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* s_x = smem;                                   // NXS slabs
    uint8_t* s_w = smem + Cfg::W;                          // NST ring stages of STG half slabs
    float* s_bias = reinterpret_cast<float*>(smem + Cfg::BIAS);
    __shared__ __align__(8) uint64_t bars[2 * NST + 2 * NXS + 5];
    __shared__ uint32_t tmem_base_s;
    const uint32_t b_wfull = smem_u32(&bars[0]), b_wempty = smem_u32(&bars[NST]);
    const uint32_t b_xfull = smem_u32(&bars[2 * NST]), b_xempty = smem_u32(&bars[2 * NST + NXS]);
    const uint32_t b_accfull = smem_u32(&bars[2 * NST + 2 * NXS]), b_accempty = b_accfull + 16;
    const uint32_t b_hready = b_accfull + 32;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#if DSP_DIR_INTERLEAVE
    // block order: (tile pair, direction, rank in pair) -- both directions of a tile run in the same wave,
    // so the second read of the layer's input image mostly hits L2
    const int dir = IS_FC ? 0 : (int)((blockIdx.x >> 1) & 1u);
    const int tile = IS_FC ? (int)blockIdx.x : (int)(((blockIdx.x >> 2) << 1) | (blockIdx.x & 1u));
#else
    const int tile = blockIdx.x, dir = IS_FC ? 0 : blockIdx.y;
#endif
    const int T = p.T;
    const uint32_t crank = cluster_ctarank();              // 0 = leader

    if (tid == 0) {
        // barriers the leader's MMA thread waits on collect one arrival per CTA
        const uint32_t both = crank == 0 ? 2u : 1u;
        for (int i = 0; i < NST; ++i) { mbar_init(b_wfull + 8 * i, both); mbar_init(b_wempty + 8 * i, 1); }
        for (int i = 0; i < NXS; ++i) { mbar_init(b_xfull + 8 * i, both); mbar_init(b_xempty + 8 * i, 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(b_accfull + 8 * i, 1); mbar_init(b_accempty + 8 * i, 2 * EPI_WARPS); }
        mbar_init(b_hready, 2 * EPI_WARPS);
        mbar_fence_init();
    }
    if (warp == 3) tmem_alloc_pair(smem_u32(&tmem_base_s), 512);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                          // the peer's barriers exist before anything lands on them
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    griddep_launch_dependents();                 // the next kernel of the stream may take SMs as this grid drains
    const uint32_t t_acc = tmem;                 // two accumulators: columns [0,128) and [128,256)
    const uint32_t t_h = tmem + 256;             // two h buffers of H/2 columns at +0 and +128

    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
        if (warp == 0) {
            // ---- weight producer: this CTA's half slabs, linear in stream order -----------------------
            if (elect_one()) {
                const size_t total = (size_t)(MODE == MODE_HEAD ? T : 1) * W_STEP;
                const uint8_t* wsrc = p.w_img + ((size_t)dir * 2 + crank) * total * HSLAB_BYTES;
                uint32_t stage = 0, phase = 0;
                for (int step = 0; step < T; ++step) {
                    // MODE_HEAD walks T passes over different weight images (split-precision terms)
                    const uint8_t* src = wsrc + (size_t)(MODE == MODE_HEAD ? step : 0) * W_STEP * HSLAB_BYTES;
                    for (int s = 0; s < W_STEP; s += STG) {
                        mbar_wait(b_wempty + 8 * stage, phase ^ 1);
                        mbar_arrive_expect_tx(b_wfull + 8 * stage, STG * HSLAB_BYTES);
                        bulk_g2s(smem_u32(s_w + (size_t)stage * STG * HSLAB_BYTES), src, STG * HSLAB_BYTES, b_wfull + 8 * stage);
                        src += (size_t)STG * HSLAB_BYTES;
                        if (++stage == NST) { stage = 0; phase ^= 1; }
                    }
                }
            }
        } else if (warp == 2) {
            // ---- x_t slab producer ------------------------------------------------------------
            if (elect_one()) {
                griddep_wait();              // the layer input is the previous kernel's output
                for (int step = 0; step < T; ++step) {
                    const int t = dir ? (T - 1 - step) : step;
                    // MODE_HEAD: pass 0 and 2 read the hi image, pass 1 the lo image of [h_fwd | h_bwd]
                    const uint8_t* xsrc = (MODE == MODE_HEAD)
                        ? p.x_img + ((size_t)tile * 2 + (step == 1 ? 1 : 0)) * KSX * SLAB_BYTES
                        : p.x_img + ((size_t)tile * T + t) * KSX * SLAB_BYTES;
                    const int xbuf = step % XB, xround = step / XB;
                    for (int j = 0; j < KSX; ++j) {
                        const int xi = xbuf * KSX + j;
                        mbar_wait(b_xempty + 8 * xi, (xround & 1) ^ 1);
                        mbar_arrive_expect_tx(b_xfull + 8 * xi, SLAB_BYTES);
                        bulk_g2s(smem_u32(s_x + (size_t)xi * SLAB_BYTES), xsrc + (size_t)j * SLAB_BYTES, SLAB_BYTES, b_xfull + 8 * xi);
                    }
                }
            }
        } else if (warp == 1 && crank != 0) {
            // ---- peer relay: forward "my half landed" to the leader's barriers, in consumption order --
            const uint32_t r_wfull = mapa_u32(b_wfull, 0), r_xfull = mapa_u32(b_xfull, 0);
            uint32_t stage = 0, phase = 0;
            for (int step = 0; step < T; ++step) {
                for (int j = 0; j < KSX; ++j) {
                    const int xi = (step % XB) * KSX + j;
                    mbar_wait(b_xfull + 8 * xi, (step / XB) & 1);
                    if (lane == 0) mbar_arrive_cluster(r_xfull + 8 * xi);
                }
                for (int s = 0; s < W_STEP; s += STG) {
                    mbar_wait(b_wfull + 8 * stage, phase);
                    if (lane == 0) mbar_arrive_cluster(r_wfull + 8 * stage);
                    if (++stage == NST) { stage = 0; phase ^= 1; }
                }
            }
        } else if (warp == 1) {
            // ---- MMA issuer (leader CTA): the whole warp walks the schedule (warp-uniform control flow
            // keeps the descriptors in uniform registers); one elected lane issues tcgen05.mma / commit --
            const bool leader = elect_one();
            const uint32_t a_lo0 = smem_desc_lo(smem_u32(s_x)), b_lo0 = smem_desc_lo(smem_u32(s_w));
            const int xk16 = p.xk16;
            uint32_t stage = 0, phase = 0, in_stage = 0;
            // half slab to consume next: wait for its stage when entering one; returns its descriptor
            auto w_acquire = [&]() -> uint32_t {
                if (in_stage == 0) { mbar_wait_cluster(b_wfull + 8 * stage, phase); tc_fence_after(); }
                return b_lo0 + (stage * STG + in_stage) * (uint32_t)(HSLAB_BYTES >> 4);
            };
            auto w_release = [&]() {
                if (++in_stage == STG) {
                    if (leader) mma2_commit(b_wempty + 8 * stage, PAIR_MASK);
                    in_stage = 0;
                    if (++stage == NST) { stage = 0; phase ^= 1; }
                }
                __syncwarp();
            };
            // x part of one chunk: A = x_t slabs in shared memory (both CTAs, own tile each)
            auto issue_x = [&](uint32_t acc, bool fresh, bool first_use, bool last_use, int step) {
#pragma unroll
                for (int j = 0; j < KSX; ++j) {
                    const int xi = (step % XB) * KSX + j;
                    if (first_use) { mbar_wait_cluster(b_xfull + 8 * xi, (step / XB) & 1); tc_fence_after(); }
                    const uint32_t bl = w_acquire();
                    if (leader) {
                        const uint32_t al = a_lo0 + (uint32_t)xi * (SLAB_BYTES >> 4);
                        const int nk = (KSX * 4 == xk16) ? 4 : min(4, xk16 - 4 * j);
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            if (k < nk) {
                                if (j == 0 && k == 0 && fresh) mma2_ss_lo<0>(acc, al, bl, IDESC);
                                else mma2_ss_lo<1>(acc, al + k * 2, bl + k * 2, IDESC);
                            }
                        }
                        if (last_use) mma2_commit(b_xempty + 8 * xi, PAIR_MASK);
                    }
                    w_release();
                }
            };
            for (int step = 0; step < T; ++step) {
                if constexpr (MODE == MODE_LSTM) {
                    const uint32_t a_t = t_h + (uint32_t)(step & 1) * 128u;
                    for (int pr = 0; pr < NCH / 2; ++pr) {
                        const uint32_t use = (uint32_t)(step * (NCH / 2) + pr);
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            mbar_wait_cluster(b_accempty + 8 * e, (use & 1u) ^ 1u);
                            tc_fence_after();
                            issue_x(t_acc + e * 128u, true, pr == 0 && e == 0, pr == NCH / 2 - 1 && e == 1, step);
                        }
                        if (pr == 0) { mbar_wait_cluster(b_hready, step & 1); tc_fence_after(); }
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
#pragma unroll
                            for (int j = 0; j < KSH; ++j) {
                                const uint32_t bl = w_acquire();
                                if (leader) {
#pragma unroll
                                    for (int k = 0; k < 4; ++k)
                                        mma2_ts_lo<1>(t_acc + e * 128u, a_t + (uint32_t)(j * 32 + k * 8), bl + k * 2, IDESC);
                                }
                                w_release();
                            }
                            if (leader) mma2_commit(b_accfull + 8 * e, PAIR_MASK);
                            __syncwarp();
                        }
                    }
                } else {
                    for (int ch = 0; ch < NCH; ++ch) {
                        // MODE_HEAD: chunk ch accumulates into buffer ch over all T passes
                        const uint32_t g = (MODE == MODE_HEAD) ? (uint32_t)ch : (uint32_t)(step * NCH + ch);
                        const uint32_t buf = g & 1u, use = g >> 1;
                        const bool fresh = (MODE != MODE_HEAD) || step == 0;
                        if (MODE != MODE_HEAD) { mbar_wait_cluster(b_accempty + 8 * buf, (use & 1u) ^ 1u); tc_fence_after(); }
                        issue_x(t_acc + buf * 128u, fresh, ch == 0, ch == NCH - 1, step);
                        if (leader && (MODE != MODE_HEAD || step == T - 1)) mma2_commit(b_accfull + 8 * buf, PAIR_MASK);
                        __syncwarp();
                    }
                }
            }
        }
    } else {
        // ---- epilogue warps: thread = site row ------------------------------------------------------
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
        const int ew = warp - 4;
        const int q = warp & 3;                      // TMEM lane quarter this warp may access
        const int sl = ew >> 2;                      // which CPT-column slice of the chunk's 128 columns
        const int row = q * 32 + lane;
        const int64_t site = (int64_t)tile * TILE + row;
        const bool valid = site < p.n;
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        // "accumulator drained" / "h written" go to the leader's barriers
        const uint32_t r_accempty = mapa_u32(b_accempty, 0), r_hready = mapa_u32(b_hready, 0);

        for (int i = tid - 128; i < NBIAS; i += EPI_WARPS * 32) s_bias[i] = p.bias[(size_t)dir * NBIAS + i];
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");           // the epilogue warps only

        if constexpr (MODE == MODE_HEAD) {
            // z = relu(fc1(x)); logits = fc2(z); probs = softmax(logits).  Each thread owns 64 of the
            // NOUT fc1 columns of its site per chunk and accumulates its share of the fc2 dot products;
            // the two column halves of a site meet through shared memory.
            __shared__ float head_part[EPI_WARPS / 4][TILE][HEAD_MAX_CLASSES];
            const int C = p.num_classes;
            float part_sum[HEAD_MAX_CLASSES];
#pragma unroll
            for (int cc = 0; cc < HEAD_MAX_CLASSES; ++cc) part_sum[cc] = 0.f;
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch) {
                const uint32_t buf = (uint32_t)ch & 1u, use = (uint32_t)ch >> 1;
                mbar_wait(b_accfull + 8 * buf, use & 1u);
                tc_fence_after();
                uint32_t v[32];
                tmem_ld32(t_acc + buf * 128u + lane_addr + (uint32_t)(sl * CPT), v);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int col = ch * 128 + sl * CPT + j;
                    const float z = fmaxf(__uint_as_float(v[j]) + s_bias[col], 0.f);
#pragma unroll
                    for (int cc = 0; cc < HEAD_MAX_CLASSES; ++cc)
                        if (cc < C) part_sum[cc] = fmaf(z, __ldg(p.w2t + (size_t)col * C + cc), part_sum[cc]);
                }
            }
#pragma unroll
            for (int cc = 0; cc < HEAD_MAX_CLASSES; ++cc) head_part[sl][row][cc] = part_sum[cc];
            asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
            if (sl == 0 && valid) {
                float lg[HEAD_MAX_CLASSES];
                float mx = -3.0e38f;
                int arg = 0;
#pragma unroll
                for (int cc = 0; cc < HEAD_MAX_CLASSES; ++cc) {
                    lg[cc] = 0.f;
                    if (cc < C) {
                        float a = __ldg(p.b2 + cc);
#pragma unroll
                        for (int s4 = 0; s4 < EPI_WARPS / 4; ++s4) a += head_part[s4][row][cc];
                        lg[cc] = a;
                        if (lg[cc] > mx) { mx = lg[cc]; arg = cc; }
                    }
                }
                float sum = 0.f;
#pragma unroll
                for (int cc = 0; cc < HEAD_MAX_CLASSES; ++cc) if (cc < C) sum += expf(lg[cc] - mx);
#pragma unroll
                for (int cc = 0; cc < HEAD_MAX_CLASSES; ++cc)
                    if (cc < C) {
                        p.logits[site * C + cc] = lg[cc];
                        p.probs[site * C + cc] = expf(lg[cc] - mx) / sum;
                    }
                if (p.labels) p.labels[site] = arg;
            }
        } else if constexpr (MODE == MODE_FC) {
            for (int step = 0; step < T; ++step) {
                uint8_t* ybase = p.y_img + ((size_t)tile * T + step) * p.y_slabs * SLAB_BYTES;
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    const uint32_t g = (uint32_t)(step * NCH + ch);
                    const uint32_t buf = g & 1u, use = g >> 1;
                    mbar_wait(b_accfull + 8 * buf, use & 1u);
                    tc_fence_after();
                    const int col0 = p.y_col_off + ch * 128 + sl * CPT;       // multiple of 32
                    uint8_t* yslab = ybase + (size_t)(col0 >> 6) * SLAB_BYTES + row * SLAB_ROW_BYTES;
                    uint32_t v[32];
                    tmem_ld32(t_acc + buf * 128u + lane_addr + (uint32_t)(sl * CPT), v);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_cluster(r_accempty + 8 * buf);
                    const float* bs = s_bias + ch * 128 + sl * CPT;
#pragma unroll
                    for (int c8 = 0; c8 < 4; ++c8) {
                        uint32_t o[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int j = c8 * 8 + e * 2;
                            const float a = fmaxf(__uint_as_float(v[j]) + bs[j], 0.f);
                            const float b = fmaxf(__uint_as_float(v[j + 1]) + bs[j + 1], 0.f);
                            o[e] = pack_half2(a, b);
                        }
                        const int chunk = ((col0 & 63) >> 3) + c8;
                        *reinterpret_cast<uint4*>(yslab + ((chunk ^ (row & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
                    }
                }
            }
        } else {
            float2 c2[NCH][UPT / 2];                  // cell state, fp32, in registers for all T steps
            // initial states: c0 -> registers, h0 -> TMEM h buffer 0 (packed FP16 pairs)
            const bool draw = p.h0 == nullptr;
            const uint64_t gs = (uint64_t)(p.site_base + site);
            const uint32_t k0 = (uint32_t)p.seed, k1 = (uint32_t)(p.seed >> 32);
            const uint32_t slot0 = (p.rng_slot + (uint32_t)dir) << 16;
            if (draw) {
                // drawn here (Philox).  Only h0 is needed before the first MMA: a compact loop stores it
                // straight into the TMEM operand buffer; c0 follows after the MMA warp has been released.
#pragma unroll 1
                for (int i = 0; i < NCH * (UPT / 4); ++i) {
                    const int unit = (i / (UPT / 4)) * 32 + sl * UPT + (i % (UPT / 4)) * 4;
                    const float4 hq = philox_normal4((uint32_t)gs, (uint32_t)(gs >> 32), slot0 | (uint32_t)(unit >> 2), p.rng_call, k0, k1);
                    tmem_st2(t_h + lane_addr + (uint32_t)(unit >> 1), pack_half2(hq.x, hq.y), pack_half2(hq.z, hq.w));
                }
                tmem_st_wait();
            } else {
                const float* h0 = p.h0 + (size_t)dir * p.state_dir_stride + (size_t)site * H;
                const float* c0 = p.c0 + (size_t)dir * p.state_dir_stride + (size_t)site * H;
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    const int u0 = ch * 32 + sl * UPT;
                    float4 cv0 = make_float4(0.f, 0.f, 0.f, 0.f), cv1 = cv0, hq0 = cv0, hq1 = cv0;
                    if (valid) {
                        cv0 = *reinterpret_cast<const float4*>(c0 + u0); cv1 = *reinterpret_cast<const float4*>(c0 + u0 + 4);
                        hq0 = *reinterpret_cast<const float4*>(h0 + u0); hq1 = *reinterpret_cast<const float4*>(h0 + u0 + 4);
                    }
                    c2[ch][0] = make_float2(cv0.x, cv0.y); c2[ch][1] = make_float2(cv0.z, cv0.w);
                    c2[ch][2] = make_float2(cv1.x, cv1.y); c2[ch][3] = make_float2(cv1.z, cv1.w);
                    tmem_st4(t_h + lane_addr + (uint32_t)(u0 >> 1), pack_half2(hq0.x, hq0.y), pack_half2(hq0.z, hq0.w),
                             pack_half2(hq1.x, hq1.y), pack_half2(hq1.z, hq1.w));
                }
                tmem_st_wait();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(r_hready);
            if (draw) {
                // c0 while the first MMAs run: parked as packed FP16 pairs in THIS thread's columns of h
                // buffer 1 (nobody touches them before this thread writes h_1 there), then read back with
                // static register indices.  (A random N(0,1) draw rounded to FP16 is as good a draw.)
                const uint32_t t_park = t_h + 128u + lane_addr;
#pragma unroll 1
                for (int i = 0; i < NCH * (UPT / 4); ++i) {
                    const int unit = (i / (UPT / 4)) * 32 + sl * UPT + (i % (UPT / 4)) * 4;
                    const float4 cv = philox_normal4((uint32_t)gs, (uint32_t)(gs >> 32), slot0 | (uint32_t)(unit >> 2) | 0x8000u, p.rng_call, k0, k1);
                    tmem_st2(t_park + (uint32_t)(unit >> 1), pack_half2(cv.x, cv.y), pack_half2(cv.z, cv.w));
                }
                tmem_st_wait();
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    uint32_t v[4];
                    tmem_ld4(t_park + (uint32_t)((ch * 32 + sl * UPT) >> 1), v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < UPT / 2; ++j) {
                        const __half2 hh = *reinterpret_cast<const __half2*>(&v[j]);
                        c2[ch][j] = make_float2(__low2float(hh), __high2float(hh));
                    }
                }
            }
            const uint32_t s_bias_u32 = smem_u32(s_bias) + (uint32_t)(sl * CPT * 4);
            for (int step = 0; step < T; ++step) {
                const int t = dir ? (T - 1 - step) : step;
                const bool last = (step == T - 1);
                uint8_t* ybase = p.y_img + ((size_t)tile * (p.write_y == 2 ? 2 : T) + (p.write_y == 2 ? 0 : t)) * p.y_slabs * SLAB_BYTES
                                 + row * SLAB_ROW_BYTES;
                const bool do_write = p.write_y == 1 || (p.write_y == 2 && last);
                const uint32_t t_hnext = t_h + (uint32_t)((step + 1) & 1) * 128u + lane_addr;
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    const uint32_t buf = (uint32_t)ch & 1u;                   // chunk pair (c, c+1) -> buffers 0, 1
                    const uint32_t use = (uint32_t)(step * (NCH / 2) + (ch >> 1));
                    mbar_wait(b_accfull + 8 * buf, use & 1u);
                    tc_fence_after();
                    const int u0 = ch * 32 + sl * UPT;
                    float2 h2[UPT / 2];
                    // PW accumulator columns (PW/8 unit pairs) are in flight per thread at a time: the whole
                    // 32-column slice where registers allow (hidden 128: 32 cell-state registers), half otherwise
                    constexpr int PW = (H == 128 || DSP_PW32_ALL) ? 32 : 16;
#pragma unroll
                    for (int part = 0; part < CPT / PW; ++part) {
                        uint32_t v[PW];
                        if constexpr (PW == 32) tmem_ld32(t_acc + buf * 128u + lane_addr + (uint32_t)(sl * CPT), reinterpret_cast<uint32_t(&)[32]>(v));
                        else tmem_ld16(t_acc + buf * 128u + lane_addr + (uint32_t)(sl * CPT + part * 16), reinterpret_cast<uint32_t(&)[16]>(v));
                        // biases of this part's units (warp-wide broadcast reads) while the TMEM load is in flight
                        float4 bq[PW / 4];
#pragma unroll
                        for (int i = 0; i < PW / 4; ++i) bq[i] = lds128(s_bias_u32 + (uint32_t)((ch * 128 + part * PW + i * 4) * 4));
                        tmem_ld_wait();
                        if (part == CPT / PW - 1) {
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive_cluster(r_accempty + 8 * buf);
                        }
#pragma unroll
                        for (int qq = 0; qq < PW / 8; ++qq) {
                            // columns of one unit pair: i i' f f' g g' o o'
                            const float4 b0 = bq[2 * qq], b1 = bq[2 * qq + 1];
                            const float2 ai = add2(make_float2(__uint_as_float(v[qq * 8 + 0]), __uint_as_float(v[qq * 8 + 1])), make_float2(b0.x, b0.y));
                            const float2 af = add2(make_float2(__uint_as_float(v[qq * 8 + 2]), __uint_as_float(v[qq * 8 + 3])), make_float2(b0.z, b0.w));
                            const float2 ag = add2(make_float2(__uint_as_float(v[qq * 8 + 4]), __uint_as_float(v[qq * 8 + 5])), make_float2(b1.x, b1.y));
                            const float2 ao = add2(make_float2(__uint_as_float(v[qq * 8 + 6]), __uint_as_float(v[qq * 8 + 7])), make_float2(b1.z, b1.w));
                            lstm_cell2<(H == 128) ? DSP_POLY_MASK_BRANCH : (KSX == 4 ? DSP_POLY_MASK_L0 : DSP_POLY_MASK)>(ai, af, ag, ao, c2[ch][part * (PW / 8) + qq], h2[part * (PW / 8) + qq]);
                        }
                    }
                    uint32_t pk[UPT / 2];
#pragma unroll
                    for (int j = 0; j < UPT / 2; ++j) pk[j] = pack_half2(h2[j].x, h2[j].y);
                    tmem_st4(t_hnext + (uint32_t)(u0 >> 1), pk[0], pk[1], pk[2], pk[3]);
                    if (do_write) {
                        const int col = dir * H + u0;                          // multiple of 8
                        uint8_t* yslab = ybase + (size_t)(col >> 6) * SLAB_BYTES;
                        const int chunk = (col & 63) >> 3;
                        *reinterpret_cast<uint4*>(yslab + (((chunk) ^ (row & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                        if (p.write_y == 2) {
                            // second image: FP16 residuals h - fp16(h), so the head sees h to ~22 bits
                            uint32_t lo[UPT / 2];
#pragma unroll
                            for (int j = 0; j < UPT / 2; ++j) {
                                const __half2 hh = *reinterpret_cast<const __half2*>(&pk[j]);
                                lo[j] = pack_half2(h2[j].x - __low2float(hh), h2[j].y - __high2float(hh));
                            }
                            uint8_t* lslab = yslab + (size_t)p.y_slabs * SLAB_BYTES;
                            *reinterpret_cast<uint4*>(lslab + (((chunk) ^ (row & 7)) << 4)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                        }
                    }
                    if (last && p.hfinal != nullptr && valid) {
                        float* hf = p.hfinal + (size_t)site * (2 * H) + dir * H + u0;
#pragma unroll
                        for (int j = 0; j < UPT / 2; j += 2)
                            *reinterpret_cast<float4*>(hf + 2 * j) = make_float4(h2[j].x, h2[j].y, h2[j + 1].x, h2[j + 1].y);
                    }
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(r_hready);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                          // no CTA leaves while the pair may still touch it
    if (warp == 3) tmem_dealloc_pair(tmem, 512);
}

// ---------------------------------------------------------------------------------------------
// Branch layers of both_bilstm (lstm_seq / lstm_signal: hidden 128, K = 16 + 128).  Their MMAs are
// tiny, so a single (tile, direction) recurrence leaves the SM waiting on its own dependency chain
// (MMA -> gate math -> h -> MMA) most of the time.  Here a CTA pair runs BOTH directions of its two
// tiles as two independent chains that fill each other's bubbles: 64-column chunks (16 hidden
// units) so that two chains fit in TMEM (per chain 2 x 64 accumulator columns + 2 x 64 h columns),
// 8 epilogue warps per chain, one MMA issuer alternating between the chains.  Everything else
// (CTA pair, half-operand staging, barrier protocol) is as in layer_kernel.
constexpr int BR_H = 128, BR_NW = 64, BR_NCH = BR_H / 16, BR_KSH = BR_H / 64;
constexpr int BR_KSX = 1;                                 // x slabs per step: only a branch's first layer (K <= 64) runs here
constexpr int BR_YS = 2 * BR_H / 64;                      // slabs of a y row [h_fwd | h_bwd] (also the K of the fused fc)
constexpr int QSLAB_BYTES = 32 * SLAB_ROW_BYTES;          // 4 KB: one CTA's share (32 rows) of a 64-column B slab
constexpr int BR_STG = 4, BR_NST = 6;                     // ring: 6 stages of 16 KB
constexpr int BR_PAIR_UNITS = 4 * BR_KSX + 4 * BR_KSH;    // X(0,c) X(0,c+1) X(1,c) X(1,c+1) H(0,c) H(0,c+1) H(1,c) H(1,c+1)
constexpr int BR_W_STEP = (BR_NCH / 2) * BR_PAIR_UNITS;   // ring units streamed per step
constexpr int BR_NBIAS = 2 * BR_NCH * BR_NW;
static_assert(BR_W_STEP % BR_STG == 0, "a step must be a whole number of ring stages");

// Dynamic shared memory of the branch kernels, as offsets from its 1 KB-aligned base: x slabs [dir][BR_KSX] at 0,
// the weight ring, the LSTM biases.  FC_TAIL adds the fc weights and biases, resident for the whole kernel, and
// double-buffers y(t) over the x + ring space, which the recurrence has finished with by then.
template <bool FC_TAIL> struct BranchSmem {
    static constexpr size_t W = (size_t)2 * BR_KSX * SLAB_BYTES;
    static constexpr size_t WFC = W + (size_t)BR_NST * BR_STG * QSLAB_BYTES;
    static constexpr size_t BIAS = WFC + (FC_TAIL ? (size_t)BR_YS * HSLAB_BYTES : 0);
    static constexpr size_t FCB = BIAS + (size_t)BR_NBIAS * sizeof(float);
    static constexpr size_t BYTES = FCB + (FC_TAIL ? 128 * sizeof(float) : 0) + 1024;     // + the alignment slack
    static_assert(!FC_TAIL || WFC == (size_t)2 * BR_YS * SLAB_BYTES, "tail A buffers alias x + ring exactly");
};

// One hidden-128 bidirectional layer, as the two-chain recurrence reads it.
struct BranchLayer {
    const uint8_t* x_img;      // [tiles][T][BR_KSX] slabs
    const uint8_t* w_img;      // [cta rank][stream unit] quarter slabs (TcLstmPack::w_img_dual)
    const float* bias;         // [dir][BR_NCH * 64] in chunk column order
    const float* h0;           // [dir][n][128] fp32; null: draw N(0,1) in-kernel (Philox)
    const float* c0;
    int64_t state_dir_stride;
    uint32_t rng_slot;         // state slot id of this layer, dir is added in-kernel
    int xk16;
    uint8_t* y_img;            // [tiles][T][BR_YS] slabs: [h_fwd | h_bwd] of every t
    uint64_t seed;
    uint32_t rng_call;
    int64_t site_base;
    int64_t n;
    int T;
};

// The per-timestep dense layer branch_fused_kernel runs behind the recurrence: relu(y(t) W^T + b), N = 128.
struct FcTail {
    const uint8_t* w_img;      // [cta rank][BR_YS] half slabs (TcDensePack layout)
    const float* bias;         // 128 floats
    uint8_t* y_img;            // [tiles][T][4] slabs
    int col0;                  // first column of y_img this layer writes
};

// The two-chain recurrence of one CTA pair, the body of both branch_kernel and branch_fused_kernel (the entry points
// only pick the layer and the tile).  FC_TAIL adds the fc tail phase of branch_fused_kernel and nothing else: the fc
// weight preload, the tail barriers and their relay, the y(t) read-back over the x + ring space, the fc MMAs and the
// fence.proxy.async + relu epilogue.
template <bool FC_TAIL>
__device__ __forceinline__ void branch_body(const BranchLayer& L, const FcTail& fc, const int tile) {
    using S = BranchSmem<FC_TAIL>;
    constexpr uint32_t IDESC = make_idesc_f16(256, BR_NW);
    constexpr uint32_t IDESC_FC = make_idesc_f16(256, 128);

    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* s_x = smem;                                   // [dir][BR_KSX] slabs          } recurrent phase
    uint8_t* s_w = smem + S::W;                            // weight ring                  }
    uint8_t* s_a = smem;                                   // tail: 2 x BR_YS slabs of y(t), aliasing the two above
    uint8_t* s_wfc = smem + S::WFC;                        // tail: this CTA's half of the fc weights (BR_YS half slabs)
    float* s_bias = reinterpret_cast<float*>(smem + S::BIAS);
    float* s_fcb = reinterpret_cast<float*>(smem + S::FCB);
    __shared__ __align__(8) uint64_t bars[2 * BR_NST + 4 * BR_KSX + 10 + (FC_TAIL ? 10 : 0)];
    __shared__ uint32_t tmem_base_s;
    const uint32_t b_wfull = smem_u32(&bars[0]), b_wempty = smem_u32(&bars[BR_NST]);
    const uint32_t b_xfull = smem_u32(&bars[2 * BR_NST]), b_xempty = b_xfull + 8 * 2 * BR_KSX;    // [dir][BR_KSX]
    const uint32_t b_accfull = b_xempty + 8 * 2 * BR_KSX, b_accempty = b_accfull + 32;            // [dir][2]
    const uint32_t b_hready = b_accempty + 32;                                                  // [dir]
    const uint32_t b_tail = b_hready + 16;                 // all epilogue warps of THIS CTA are past the last y store
    const uint32_t b_wfc = b_tail + 8;                     // fc weights landed (both CTAs)
    const uint32_t b_afull = b_wfc + 8, b_aempty = b_afull + 16;                                  // [2]
    const uint32_t b_faccfull = b_aempty + 16, b_faccempty = b_faccfull + 16;                     // [2]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int T = L.T;
    const uint32_t crank = cluster_ctarank();

    if (tid == 0) {
        const uint32_t both = crank == 0 ? 2u : 1u;
        for (int i = 0; i < BR_NST; ++i) { mbar_init(b_wfull + 8 * i, both); mbar_init(b_wempty + 8 * i, 1); }
        for (int i = 0; i < 2 * BR_KSX; ++i) { mbar_init(b_xfull + 8 * i, both); mbar_init(b_xempty + 8 * i, 1); }
        for (int i = 0; i < 4; ++i) { mbar_init(b_accfull + 8 * i, 1); mbar_init(b_accempty + 8 * i, EPI_WARPS); }   // 8 warps x 2 CTAs
        for (int i = 0; i < 2; ++i) mbar_init(b_hready + 8 * i, EPI_WARPS);
        if constexpr (FC_TAIL) {
            mbar_init(b_tail, EPI_WARPS);
            mbar_init(b_wfc, both);
            for (int i = 0; i < 2; ++i) {
                mbar_init(b_afull + 8 * i, both); mbar_init(b_aempty + 8 * i, 1);
                mbar_init(b_faccfull + 8 * i, 1); mbar_init(b_faccempty + 8 * i, 2 * EPI_WARPS);
            }
        }
        mbar_fence_init();
    }
    if (warp == 3) tmem_alloc_pair(smem_u32(&tmem_base_s), 512);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem = tmem_base_s;
    griddep_launch_dependents();
    // chain d: accumulators at d*128 + {0, 64}, h buffers at 256 + d*128 + {0, 64}
    auto t_acc = [&](int d, int e) -> uint32_t { return tmem + (uint32_t)(d * 128 + e * 64); };
    auto t_h = [&](int d, int b) -> uint32_t { return tmem + 256u + (uint32_t)(d * 128 + b * 64); };

    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
        if (warp == 0) {
            if (elect_one()) {
                if constexpr (FC_TAIL) {
                    // fc weights first: they stay put for the whole kernel
                    mbar_arrive_expect_tx(b_wfc, BR_YS * HSLAB_BYTES);
                    bulk_g2s(smem_u32(s_wfc), fc.w_img + (size_t)crank * BR_YS * HSLAB_BYTES, BR_YS * HSLAB_BYTES, b_wfc);
                }
                const uint8_t* wsrc = L.w_img + (size_t)crank * BR_W_STEP * QSLAB_BYTES;
                uint32_t stage = 0, phase = 0;
                for (int step = 0; step < T; ++step) {
                    const uint8_t* src = wsrc;
                    for (int s = 0; s < BR_W_STEP; s += BR_STG) {
                        mbar_wait(b_wempty + 8 * stage, phase ^ 1);
                        mbar_arrive_expect_tx(b_wfull + 8 * stage, BR_STG * QSLAB_BYTES);
                        bulk_g2s(smem_u32(s_w + (size_t)stage * BR_STG * QSLAB_BYTES), src, BR_STG * QSLAB_BYTES, b_wfull + 8 * stage);
                        src += (size_t)BR_STG * QSLAB_BYTES;
                        if (++stage == BR_NST) { stage = 0; phase ^= 1; }
                    }
                }
            }
        } else if (warp == 2) {
            if (elect_one()) {
                griddep_wait();              // the layer input is the previous kernel's output
                for (int step = 0; step < T; ++step)
                    for (int d = 0; d < 2; ++d) {
                        const int t = d ? (T - 1 - step) : step;
                        const uint8_t* xsrc = L.x_img + ((size_t)tile * T + t) * BR_KSX * SLAB_BYTES;
                        for (int j = 0; j < BR_KSX; ++j) {
                            const uint32_t o = 8u * (uint32_t)(d * BR_KSX + j);
                            mbar_wait(b_xempty + o, (step & 1) ^ 1);
                            mbar_arrive_expect_tx(b_xfull + o, SLAB_BYTES);
                            bulk_g2s(smem_u32(s_x + (size_t)(d * BR_KSX + j) * SLAB_BYTES), xsrc + (size_t)j * SLAB_BYTES, SLAB_BYTES, b_xfull + o);
                        }
                    }
                if constexpr (FC_TAIL) {
                    // ---- tail: y(t) of the own tile back from L2, double buffered over the idle x + ring space ----
                    mbar_wait(b_tail, 0);    // every y store of this CTA is done and fenced towards the async proxy;
                                             // it also implies all recurrent MMAs (the last readers of x + ring) completed
                    for (int t = 0; t < T; ++t) {
                        const uint32_t buf = (uint32_t)t & 1u;
                        mbar_wait(b_aempty + 8 * buf, ((uint32_t)(t >> 1) & 1u) ^ 1u);
                        mbar_arrive_expect_tx(b_afull + 8 * buf, BR_YS * SLAB_BYTES);
                        bulk_g2s(smem_u32(s_a + (size_t)buf * BR_YS * SLAB_BYTES), L.y_img + ((size_t)tile * T + t) * BR_YS * SLAB_BYTES,
                                 BR_YS * SLAB_BYTES, b_afull + 8 * buf);
                    }
                }
            }
        } else if (warp == 1 && crank != 0) {
            const uint32_t r_wfull = mapa_u32(b_wfull, 0), r_xfull = mapa_u32(b_xfull, 0);
            uint32_t stage = 0, phase = 0;
            for (int step = 0; step < T; ++step) {
                for (int i = 0; i < 2 * BR_KSX; ++i) {
                    mbar_wait(b_xfull + 8 * i, step & 1);
                    if (lane == 0) mbar_arrive_cluster(r_xfull + 8 * i);
                }
                for (int s = 0; s < BR_W_STEP; s += BR_STG) {
                    mbar_wait(b_wfull + 8 * stage, phase);
                    if (lane == 0) mbar_arrive_cluster(r_wfull + 8 * stage);
                    if (++stage == BR_NST) { stage = 0; phase ^= 1; }
                }
            }
            if constexpr (FC_TAIL) {
                const uint32_t r_wfc = mapa_u32(b_wfc, 0), r_afull = mapa_u32(b_afull, 0);
                mbar_wait(b_wfc, 0);
                if (lane == 0) mbar_arrive_cluster(r_wfc);
                for (int t = 0; t < T; ++t) {
                    const uint32_t buf = (uint32_t)t & 1u;
                    mbar_wait(b_afull + 8 * buf, (uint32_t)(t >> 1) & 1u);
                    if (lane == 0) mbar_arrive_cluster(r_afull + 8 * buf);
                }
            }
        } else if (warp == 1) {
            const bool leader = elect_one();
            const uint32_t a_lo0 = smem_desc_lo(smem_u32(s_x)), b_lo0 = smem_desc_lo(smem_u32(s_w));
            const int xk16 = L.xk16;
            uint32_t stage = 0, phase = 0, in_stage = 0;
            auto w_acquire = [&]() -> uint32_t {
                if (in_stage == 0) { mbar_wait_cluster(b_wfull + 8 * stage, phase); tc_fence_after(); }
                return b_lo0 + (stage * BR_STG + in_stage) * (uint32_t)(QSLAB_BYTES >> 4);
            };
            auto w_release = [&]() {
                if (++in_stage == BR_STG) {
                    if (leader) mma2_commit(b_wempty + 8 * stage, PAIR_MASK);
                    in_stage = 0;
                    if (++stage == BR_NST) { stage = 0; phase ^= 1; }
                }
                __syncwarp();
            };
            for (int step = 0; step < T; ++step) {
                for (int pr = 0; pr < BR_NCH / 2; ++pr) {
                    const uint32_t use = (uint32_t)(step * (BR_NCH / 2) + pr);
#pragma unroll
                    for (int d = 0; d < 2; ++d)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            mbar_wait_cluster(b_accempty + 8 * (d * 2 + e), (use & 1u) ^ 1u);
                            tc_fence_after();
#pragma unroll
                            for (int j = 0; j < BR_KSX; ++j) {
                                const uint32_t xo = 8u * (uint32_t)(d * BR_KSX + j);
                                if (pr == 0 && e == 0) { mbar_wait_cluster(b_xfull + xo, step & 1); tc_fence_after(); }
                                const uint32_t bl = w_acquire();
                                if (leader) {
                                    const uint32_t al = a_lo0 + (uint32_t)(d * BR_KSX + j) * (SLAB_BYTES >> 4);
                                    const int nk = (BR_KSX * 4 == xk16) ? 4 : min(4, xk16 - 4 * j);
#pragma unroll
                                    for (int k = 0; k < 4; ++k) {
                                        if (k < nk) {
                                            if (j == 0 && k == 0) mma2_ss_lo<0>(t_acc(d, e), al, bl, IDESC);
                                            else mma2_ss_lo<1>(t_acc(d, e), al + k * 2, bl + k * 2, IDESC);
                                        }
                                    }
                                    if (pr == BR_NCH / 2 - 1 && e == 1) mma2_commit(b_xempty + xo, PAIR_MASK);
                                }
                                w_release();
                            }
                        }
#pragma unroll
                    for (int d = 0; d < 2; ++d) {
                        if (pr == 0) { mbar_wait_cluster(b_hready + 8 * d, step & 1); tc_fence_after(); }
                        const uint32_t a_t = t_h(d, step & 1);
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
#pragma unroll
                            for (int j = 0; j < BR_KSH; ++j) {
                                const uint32_t bl = w_acquire();
                                if (leader) {
#pragma unroll
                                    for (int k = 0; k < 4; ++k)
                                        mma2_ts_lo<1>(t_acc(d, e), a_t + (uint32_t)(j * 32 + k * 8), bl + k * 2, IDESC);
                                }
                                w_release();
                            }
                            if (leader) mma2_commit(b_accfull + 8 * (d * 2 + e), PAIR_MASK);
                            __syncwarp();
                        }
                    }
                }
            }
            if constexpr (FC_TAIL) {
                // ---- tail: fc = y(t) * W_fc^T, accumulators = the (now idle) columns of chain 0 / chain 1 ----
                const uint32_t fa_lo0 = smem_desc_lo(smem_u32(s_a)), fb_lo0 = smem_desc_lo(smem_u32(s_wfc));
                mbar_wait_cluster(b_wfc, 0);
                tc_fence_after();
                for (int t = 0; t < T; ++t) {
                    const uint32_t buf = (uint32_t)t & 1u, use = (uint32_t)(t >> 1);
                    mbar_wait_cluster(b_faccempty + 8 * buf, (use & 1u) ^ 1u);
                    mbar_wait_cluster(b_afull + 8 * buf, use & 1u);
                    tc_fence_after();
                    if (leader) {
#pragma unroll
                        for (int j = 0; j < BR_YS; ++j) {
                            const uint32_t al = fa_lo0 + (buf * BR_YS + (uint32_t)j) * (SLAB_BYTES >> 4);
                            const uint32_t bl = fb_lo0 + (uint32_t)j * (HSLAB_BYTES >> 4);
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                if (j == 0 && k == 0) mma2_ss_lo<0>(tmem + buf * 128u, al, bl, IDESC_FC);
                                else mma2_ss_lo<1>(tmem + buf * 128u, al + k * 2, bl + k * 2, IDESC_FC);
                            }
                        }
                        mma2_commit(b_aempty + 8 * buf, PAIR_MASK);
                        mma2_commit(b_faccfull + 8 * buf, PAIR_MASK);
                    }
                    __syncwarp();
                }
            }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
        const int ew = warp - 4;
        const int d = ew >> 3;                       // chain = direction
        const int q = warp & 3;                      // TMEM lane quarter
        const int half = (ew >> 2) & 1;              // which 32 of the chunk's 64 columns (8 hidden units)
        const int row = q * 32 + lane;
        const int64_t site = (int64_t)tile * TILE + row;
        const bool valid = site < L.n;
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        const uint32_t r_accempty = mapa_u32(b_accempty, 0) + 16u * (uint32_t)d, r_hready = mapa_u32(b_hready, 0) + 8u * (uint32_t)d;
        const uint32_t b_myfull = b_accfull + 16u * (uint32_t)d;

        for (int i = tid - 128; i < BR_NBIAS; i += EPI_WARPS * 32) s_bias[i] = L.bias[i];
        if constexpr (FC_TAIL)
            for (int i = tid - 128; i < 128; i += EPI_WARPS * 32) s_fcb[i] = fc.bias[i];
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");

        constexpr int UPT = 8;
        float2 c2[BR_NCH][UPT / 2];
        const bool draw = L.h0 == nullptr;
        const uint64_t gs = (uint64_t)(L.site_base + site);
        const uint32_t k0 = (uint32_t)L.seed, k1 = (uint32_t)(L.seed >> 32);
        const uint32_t slot0 = (L.rng_slot + (uint32_t)d) << 16;
        if (draw) {
#pragma unroll 1
            for (int i = 0; i < BR_NCH * (UPT / 4); ++i) {
                const int unit = (i >> 1) * 16 + half * UPT + (i & 1) * 4;
                const float4 hq = philox_normal4((uint32_t)gs, (uint32_t)(gs >> 32), slot0 | (uint32_t)(unit >> 2), L.rng_call, k0, k1);
                tmem_st2(t_h(d, 0) + lane_addr + (uint32_t)(unit >> 1), pack_half2(hq.x, hq.y), pack_half2(hq.z, hq.w));
            }
            tmem_st_wait();
        } else {
            const float* h0 = L.h0 + (size_t)d * L.state_dir_stride + (size_t)site * BR_H;
            const float* c0 = L.c0 + (size_t)d * L.state_dir_stride + (size_t)site * BR_H;
#pragma unroll
            for (int ch = 0; ch < BR_NCH; ++ch) {
                const int u0 = ch * 16 + half * UPT;
                float4 cv0 = make_float4(0.f, 0.f, 0.f, 0.f), cv1 = cv0, hq0 = cv0, hq1 = cv0;
                if (valid) {
                    cv0 = *reinterpret_cast<const float4*>(c0 + u0); cv1 = *reinterpret_cast<const float4*>(c0 + u0 + 4);
                    hq0 = *reinterpret_cast<const float4*>(h0 + u0); hq1 = *reinterpret_cast<const float4*>(h0 + u0 + 4);
                }
                c2[ch][0] = make_float2(cv0.x, cv0.y); c2[ch][1] = make_float2(cv0.z, cv0.w);
                c2[ch][2] = make_float2(cv1.x, cv1.y); c2[ch][3] = make_float2(cv1.z, cv1.w);
                tmem_st4(t_h(d, 0) + lane_addr + (uint32_t)(u0 >> 1), pack_half2(hq0.x, hq0.y), pack_half2(hq0.z, hq0.w),
                         pack_half2(hq1.x, hq1.y), pack_half2(hq1.z, hq1.w));
            }
            tmem_st_wait();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(r_hready);
        if (draw) {          // c0 behind the first MMAs, parked in this thread's columns of h buffer 1 (see layer_kernel)
            const uint32_t t_park = t_h(d, 1) + lane_addr;
#pragma unroll 1
            for (int i = 0; i < BR_NCH * (UPT / 4); ++i) {
                const int unit = (i >> 1) * 16 + half * UPT + (i & 1) * 4;
                const float4 cv = philox_normal4((uint32_t)gs, (uint32_t)(gs >> 32), slot0 | (uint32_t)(unit >> 2) | 0x8000u, L.rng_call, k0, k1);
                tmem_st2(t_park + (uint32_t)(unit >> 1), pack_half2(cv.x, cv.y), pack_half2(cv.z, cv.w));
            }
            tmem_st_wait();
#pragma unroll
            for (int ch = 0; ch < BR_NCH; ++ch) {
                uint32_t v[4];
                tmem_ld4(t_park + (uint32_t)((ch * 16 + half * UPT) >> 1), v);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < UPT / 2; ++j) {
                    const __half2 hh = *reinterpret_cast<const __half2*>(&v[j]);
                    c2[ch][j] = make_float2(__low2float(hh), __high2float(hh));
                }
            }
        }
        const uint32_t s_bias_u32 = smem_u32(s_bias) + (uint32_t)((d * BR_NCH * BR_NW + half * 32) * 4);
        for (int step = 0; step < T; ++step) {
            const int t = d ? (T - 1 - step) : step;
            uint8_t* ybase = L.y_img + ((size_t)tile * T + t) * BR_YS * SLAB_BYTES + row * SLAB_ROW_BYTES;
            const uint32_t t_hnext = t_h(d, (step + 1) & 1) + lane_addr;
#pragma unroll
            for (int ch = 0; ch < BR_NCH; ++ch) {
                const int e = ch & 1;
                const uint32_t use = (uint32_t)(step * (BR_NCH / 2) + (ch >> 1));
                mbar_wait(b_myfull + 8 * e, use & 1u);
                tc_fence_after();
                const int u0 = ch * 16 + half * UPT;
                float2 h2[UPT / 2];
#pragma unroll
                for (int part = 0; part < 2; ++part) {
                    uint32_t v[16];
                    tmem_ld16(t_acc(d, e) + lane_addr + (uint32_t)(half * 32 + part * 16), v);
                    float4 bq[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) bq[i] = lds128(s_bias_u32 + (uint32_t)((ch * BR_NW + part * 16 + i * 4) * 4));
                    tmem_ld_wait();
                    if (part == 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive_cluster(r_accempty + 8 * e);
                    }
#pragma unroll
                    for (int qq = 0; qq < 2; ++qq) {
                        const float4 b0 = bq[2 * qq], b1 = bq[2 * qq + 1];
                        const float2 ai = add2(make_float2(__uint_as_float(v[qq * 8 + 0]), __uint_as_float(v[qq * 8 + 1])), make_float2(b0.x, b0.y));
                        const float2 af = add2(make_float2(__uint_as_float(v[qq * 8 + 2]), __uint_as_float(v[qq * 8 + 3])), make_float2(b0.z, b0.w));
                        const float2 ag = add2(make_float2(__uint_as_float(v[qq * 8 + 4]), __uint_as_float(v[qq * 8 + 5])), make_float2(b1.x, b1.y));
                        const float2 ao = add2(make_float2(__uint_as_float(v[qq * 8 + 6]), __uint_as_float(v[qq * 8 + 7])), make_float2(b1.z, b1.w));
                        lstm_cell2<DSP_POLY_MASK_BRANCH>(ai, af, ag, ao, c2[ch][part * 2 + qq], h2[part * 2 + qq]);
                    }
                }
                uint32_t pk[UPT / 2];
#pragma unroll
                for (int j = 0; j < UPT / 2; ++j) pk[j] = pack_half2(h2[j].x, h2[j].y);
                tmem_st4(t_hnext + (uint32_t)(u0 >> 1), pk[0], pk[1], pk[2], pk[3]);
                const int col = d * BR_H + u0;                             // multiple of 8
                uint8_t* yslab = ybase + (size_t)(col >> 6) * SLAB_BYTES;
                *reinterpret_cast<uint4*>(yslab + ((((col & 63) >> 3) ^ (row & 7)) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            }
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(r_hready);
        }
        if constexpr (FC_TAIL) {
            // ---- tail: this CTA's y image is complete; hand it to the async proxy (the bulk copies of warp 2) ----
            asm volatile("fence.proxy.async.global;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(b_tail);
            const int sl = ew >> 2;                  // 32-column slice of the 128 fc outputs
            const uint32_t r_faccempty = mapa_u32(b_faccempty, 0);
            const int col0 = fc.col0 + sl * 32;
            const float* bs = s_fcb + sl * 32;
            for (int t = 0; t < T; ++t) {
                const uint32_t buf = (uint32_t)t & 1u, use = (uint32_t)(t >> 1);
                mbar_wait(b_faccfull + 8 * buf, use & 1u);
                tc_fence_after();
                uint32_t v[32];
                tmem_ld32(tmem + buf * 128u + lane_addr + (uint32_t)(sl * 32), v);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(r_faccempty + 8 * buf);
                uint8_t* yslab = fc.y_img + (((size_t)tile * T + t) * BR_YS + (size_t)(col0 >> 6)) * SLAB_BYTES + row * SLAB_ROW_BYTES;
#pragma unroll
                for (int c8 = 0; c8 < 4; ++c8) {
                    uint32_t o[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int j = c8 * 8 + e * 2;
                        const float a = fmaxf(__uint_as_float(v[j]) + bs[j], 0.f);
                        const float b = fmaxf(__uint_as_float(v[j + 1]) + bs[j + 1], 0.f);
                        o[e] = pack_half2(a, b);
                    }
                    const int chunk = ((col0 & 63) >> 3) + c8;
                    *reinterpret_cast<uint4*>(yslab + ((chunk ^ (row & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 3) tmem_dealloc_pair(tmem, 512);
}

// The hidden-128 layers of a branch, one launch per layer (DSP_B200_BRANCH_DUAL=1, or where the wave cost favours it).
__global__ void __launch_bounds__(NTHREADS, 1)
branch_kernel(const LayerParams p) {
    branch_body<false>({p.x_img, p.w_img, p.bias, p.h0, p.c0, p.state_dir_stride, p.rng_slot, p.xk16, p.y_img,
                        p.seed, p.rng_call, p.site_base, p.n, p.T}, FcTail{}, (int)blockIdx.x);
}

// ---------------------------------------------------------------------------------------------
// both_bilstm's two branches in ONE launch, with their per-timestep dense layers fused behind them
// (models.py:196-201 and :212-217, then the concat of :225).  Grid = 2 x tile pairs of CTA pairs: cluster
// 2k runs lstm_seq + fc_seq, cluster 2k+1 lstm_signal + fc_signal for the same two site tiles, so the
// launch has one tail instead of four and both halves of a tile's lstm_comb input are produced in the same
// wave.  The recurrent phase is branch_kernel's, the same branch_body.  fc needs h_fwd(t) and
// h_bwd(t) of the same t, which the two chains produce T-1-2t steps apart, so it runs as a TAIL phase of the
// same CTA pair once step T-1 is done: the pair streams its own y image back (written minutes of
// microseconds ago by its own epilogue warps: L2 hits, no second kernel re-reading it from HBM), multiplies
// by the fc weights that have sat in shared memory since the prologue (M = 256 pair MMA, N = 128, K = 256)
// into the now idle accumulator columns, and the epilogue warps write relu(. + b) as the FP16 image of
// lstm_comb's input.  What the separate fc launches cost (two HBM-bound passes at the end of a wave that
// has nothing to overlap them with) becomes ~13 short L2-fed MMA steps per tile, overlapped across CTAs with
// other tiles' recurrent phases.
struct FusedBranchParams {
    const uint8_t* x_img[2];       // [branch] first-layer image: seq features / signal rectangle
    const uint8_t* w_img[2];       // [branch] branch_kernel weight stream
    const float* bias[2];
    const float* h0[2];            // [branch] null: Philox
    const float* c0[2];
    int64_t state_dir_stride[2];
    uint32_t rng_slot[2];
    int xk16[2];
    uint8_t* y_img[2];             // [branch] [tiles][T][4] slabs: [h_fwd | h_bwd] of every t
    const uint8_t* fcw_img[2];     // [branch] [rank][4] half slabs (TcDensePack layout)
    const float* fcb[2];           // [branch] 128 floats
    uint8_t* comb_img;             // [tiles][T][4] slabs: [relu(fc_seq) | relu(fc_signal)]
    uint64_t seed;
    uint32_t rng_call;
    int64_t site_base;
    int64_t n;
    int T;
};

__global__ void __launch_bounds__(NTHREADS, 1)
branch_fused_kernel(const FusedBranchParams p) {
    const int br = (int)((blockIdx.x >> 1) & 1u);                                   // 0 seq, 1 signal
    const int tile = (int)(((blockIdx.x >> 2) << 1) | (blockIdx.x & 1u));
    branch_body<true>({p.x_img[br], p.w_img[br], p.bias[br], p.h0[br], p.c0[br], p.state_dir_stride[br], p.rng_slot[br],
                       p.xk16[br], p.y_img[br], p.seed, p.rng_call, p.site_base, p.n, p.T},
                      {p.fcw_img[br], p.fcb[br], p.comb_img, br * 128}, tile);    // comb columns: [fc_seq | fc_signal]
}

// ---------------------------------------------------------------------------------------------
// Feature assembly into slab images (models.py:182-195): per (site, t) one row of
// [embed(kmer) | mean | std | len/32 | mean_lo | std_lo | len_lo | 0...] (seq) and of the signal
// rectangle (signal), FP16.  The three scalar features arrive as float32 of any magnitude (lens are
// raw sample counts, call_modifications.py:161): each is carried as an FP16 value plus the FP16
// residual of that rounding in a spare K column of the 16-wide image (`split`; the matching W_ih
// column is duplicated at pack time), i.e. to ~22 bits at no extra MMA; lens are pre-scaled by 2^-5
// (the weight column by 2^5) so that counts up to 2^21 stay inside the FP16 range.
constexpr float SEQ_LEN_SCALE = 1.f / 32.f;
__device__ __forceinline__ float clamp_half(float v) { return fminf(fmaxf(v, -65504.f), 65504.f); }
__device__ __forceinline__ float half_residual(float v) { return v - __half2float(__float2half_rn(v)); }

__global__ void prep_images_kernel(const float* __restrict__ kmer, const float* __restrict__ means,
                                   const float* __restrict__ stds, const float* __restrict__ lens,
                                   const float* __restrict__ signals, const float* __restrict__ embed,
                                   int E, int vocab, int use_len, int split, int S, int T, int64_t n, int64_t n_pad,
                                   uint8_t* __restrict__ xseq_img, uint8_t* __restrict__ xsig_img) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // (site, t)
    if (idx >= n_pad * T) return;
    const int64_t site = idx / T;
    const int t = (int)(idx - site * T);
    const int64_t tile = site >> 7;
    const int row = (int)(site & 127);
    const bool valid = site < n;
    const size_t slab = ((size_t)tile * T + t) * SLAB_BYTES;
    if (xseq_img) {
        float f[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) f[i] = 0.f;
        if (valid) {
            int c = 0;
            if (E > 0) {
                long long code = (long long)kmer[site * T + t];
                code = code < 0 ? 0 : (code >= vocab ? vocab - 1 : code);
                for (int e = 0; e < E && c < 16; ++e) f[c++] = embed[code * E + e];
            }
            const int nsc = use_len ? 3 : 2;
            float sc[3];
            sc[0] = clamp_half(means[site * T + t]);
            sc[1] = clamp_half(stds[site * T + t]);
            sc[2] = use_len ? clamp_half(lens[site * T + t] * (split ? SEQ_LEN_SCALE : 1.f)) : 0.f;
            for (int i = 0; i < nsc && c + i < 16; ++i) {
                f[c + i] = sc[i];
                if (split) f[c + nsc + i] = half_residual(sc[i]);
            }
        }
        uint8_t* dst = xseq_img + slab + row * SLAB_ROW_BYTES;
#pragma unroll
        for (int chunk = 0; chunk < 2; ++chunk) {
            uint4 o;
            o.x = pack_half2(f[chunk * 8 + 0], f[chunk * 8 + 1]); o.y = pack_half2(f[chunk * 8 + 2], f[chunk * 8 + 3]);
            o.z = pack_half2(f[chunk * 8 + 4], f[chunk * 8 + 5]); o.w = pack_half2(f[chunk * 8 + 6], f[chunk * 8 + 7]);
            *reinterpret_cast<uint4*>(dst + ((chunk ^ (row & 7)) << 4)) = o;
        }
    }
    if (xsig_img) {
        const float* src = signals + (site * T + t) * S;
        uint8_t* dst = xsig_img + slab + row * SLAB_ROW_BYTES;
        const int nchunk = ((S + 15) / 16) * 2;
        const bool vec = (S & 3) == 0;               // rows of the signal rectangle are 16-byte aligned: 128-bit loads
        for (int chunk = 0; chunk < nchunk; ++chunk) {
            float f[8];
            if (vec) {
#pragma unroll
                for (int h4 = 0; h4 < 2; ++h4) {
                    const int k = chunk * 8 + h4 * 4;
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (valid && k < S) v = __ldg(reinterpret_cast<const float4*>(src + k));
                    f[h4 * 4] = v.x; f[h4 * 4 + 1] = v.y; f[h4 * 4 + 2] = v.z; f[h4 * 4 + 3] = v.w;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) { const int k = chunk * 8 + i; f[i] = (valid && k < S) ? src[k] : 0.f; }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] = clamp_half(f[i]);          // an FP16 inf would turn into NaN probabilities
            uint4 o;
            o.x = pack_half2(f[0], f[1]); o.y = pack_half2(f[2], f[3]); o.z = pack_half2(f[4], f[5]); o.w = pack_half2(f[6], f[7]);
            *reinterpret_cast<uint4*>(dst + ((chunk ^ (row & 7)) << 4)) = o;
        }
    }
}

// ---- host-side packing ------------------------------------------------------------------------
// Weight images are written per CTA rank of the pair: [dir][rank][half slab in stream order], a half
// slab = the 64 B rows (gate / output columns) rank r contributes to a 128-column chunk.
struct TcLstmPack {
    uint8_t* w_img = nullptr;   // [2][2][NCH*KS] half slabs
    float* bias = nullptr;      // [2][NCH*128], scaled like the weights
    int KSX = 0, xk16 = 0;
    // hidden-128 layers also carry the branch_kernel layout (both directions in one stream, 64-column chunks)
    uint8_t* w_img_dual = nullptr;
    float* bias_dual = nullptr;
};
struct TcDensePack {
    uint8_t* w_img = nullptr;   // [2][NCH*KS] (x passes for the head) half slabs
    float* bias = nullptr;      // [NCH*128]
    int KS = 0;
};
struct TcState {
    uint8_t* xseq_img = nullptr;
    uint8_t* xsig_img = nullptr;
    uint8_t* ybuf[2] = {nullptr, nullptr};
    uint8_t* comb_img = nullptr;
    float* hfinal = nullptr;
    uint8_t* hfin_img = nullptr;   // [tiles][hi,lo][2H/64] slabs: [h_fwd(T-1) | h_bwd(0)] as FP16 hi + FP16 residual
    TcDensePack* head_pack = nullptr;
    bool tc_head = false;
    bool seq_split = false;        // scalar sequence features as FP16 value + residual columns
    bool pdl = true;               // programmatic dependent launch between the kernels of a forward
    int force_dual = -1;           // hidden-128 layers: -1 pick by wave cost, 0 layer_kernel, 1 branch_kernel
    int64_t tiles = 0;
    std::vector<TcLstmPack*> lstm_packs;
    std::vector<TcDensePack*> dense_packs;
};

// element (row n of a 128-row chunk, k within a 64-wide K slab) of stream half slab s
void put_half(std::vector<uint8_t>& img, size_t rank_base, size_t s, int n, int k, float v) {
    __half h = __float2half_rn(v);
    memcpy(&img[(rank_base + s) * HSLAB_BYTES + slab_offset_bytes((uint32_t)(n & 63), (uint32_t)k)], &h, 2);
}

int tc_alloc(Model* m, void** p, size_t bytes) {
    cudaError_t e = cudaMalloc(p, bytes ? bytes : 16);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e)); return DSP_ERR_NOMEM; }
    m->device_allocs.push_back(*p);
    return DSP_OK;
}

// CTA-pair kernels: clusters of 2 along x, programmatic dependent launch unless DSP_B200_PDL=0 turned it off.
template <class Params>
int launch_pair(Model* m, void (*kern)(Params), const Params& p, dim3 grid, size_t smem, cudaStream_t st) {
    DSP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(NTHREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = ((TcState*)m->tc_state)->pdl ? 2 : 1;
    DSP_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
    m->launches++;
    return DSP_OK;
}

template <int KSX, int H, int MODE, int NOUT>
int launch_layer(Model* m, const LayerParams& p, int64_t tiles, cudaStream_t st) {
    const unsigned tiles2 = (unsigned)((tiles + 1) / 2 * 2);                          // CTA pairs: the workspace is padded too
#if DSP_DIR_INTERLEAVE
    const dim3 grid(MODE != MODE_LSTM ? tiles2 : 2 * tiles2, 1);
#else
    const dim3 grid(tiles2, MODE != MODE_LSTM ? 1 : 2);
#endif
    return launch_pair(m, layer_kernel<KSX, H, MODE, NOUT>, p, grid, LayerCfg<KSX, H, MODE, NOUT>::BYTES, st);
}

int launch_branch(Model* m, const LayerParams& p, int64_t tiles, cudaStream_t st) {
    return launch_pair(m, branch_kernel, p, dim3((unsigned)((tiles + 1) / 2 * 2), 1), BranchSmem<false>::BYTES, st);
}

int launch_branch_fused(Model* m, const FusedBranchParams& p, int64_t tiles, cudaStream_t st) {
    // (tile pair, branch, rank in pair)
    return launch_pair(m, branch_fused_kernel, p, dim3((unsigned)(2 * ((tiles + 1) / 2 * 2)), 1), BranchSmem<true>::BYTES, st);
}

int launch_lstm(Model* m, int KSX, int H, const LayerParams& p, int64_t tiles, cudaStream_t st) {
    if (H == 128) {
        if (KSX == 1) return launch_layer<1, 128, MODE_LSTM, 0>(m, p, tiles, st);
        if (KSX == 4) return launch_layer<4, 128, MODE_LSTM, 0>(m, p, tiles, st);
    } else if (H == 256) {
        if (KSX == 1) return launch_layer<1, 256, MODE_LSTM, 0>(m, p, tiles, st);
        if (KSX == 4) return launch_layer<4, 256, MODE_LSTM, 0>(m, p, tiles, st);
        if (KSX == 8) return launch_layer<8, 256, MODE_LSTM, 0>(m, p, tiles, st);
    }
    set_error("tcgen05 path: unsupported LSTM layer shape (x slabs %d, hidden %d)", KSX, H);
    return DSP_ERR_INVALID;
}

int launch_fc(Model* m, int KS, int NOUT, const LayerParams& p, int64_t tiles, cudaStream_t st) {
    if (KS == 4 && NOUT == 128) return launch_layer<4, 0, MODE_FC, 128>(m, p, tiles, st);
    if (KS == 8 && NOUT == 256) return launch_layer<8, 0, MODE_FC, 256>(m, p, tiles, st);
    set_error("tcgen05 path: unsupported dense shape (K slabs %d, N %d)", KS, NOUT);
    return DSP_ERR_INVALID;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
int tc_create(Model* m) {
    const dsp_config& c = m->cfg;
    DSP_REQUIRE(c.hidden_size == 256, DSP_ERR_INVALID,
                "DSP_PRECISION_FP16 (tcgen05) supports hidden_size 256 (got %d); use DSP_PRECISION_FP32", c.hidden_size);
    DSP_REQUIRE(c.signal_len <= 64 && m->kseq <= 16, DSP_ERR_INVALID,
                "DSP_PRECISION_FP16 supports signal_len <= 64 and <= 16 sequence features per base");
    TcState* s = new TcState();
    m->tc_state = s;
    // Launch-strategy switches (neither changes a result) are read ONCE here, at handle creation:
    // DSP_B200_PDL=0 turns programmatic dependent launch off, DSP_B200_BRANCH_DUAL=0|1 forces which kernel
    // runs the hidden-128 layers.
    if (const char* e = getenv("DSP_B200_PDL")) s->pdl = atoi(e) != 0;
    if (const char* e = getenv("DSP_B200_BRANCH_DUAL")) s->force_dual = atoi(e) != 0;
    {
        const int e = c.is_base ? c.embedding_size : 0, nsc = c.is_signallen ? 3 : 2;
        s->seq_split = c.module != DSP_SIGNAL_BILSTM && e + 2 * nsc <= 16;
    }
    s->tiles = ((m->cap + TILE - 1) / TILE + 1) / 2 * 2;     // whole CTA pairs
    const size_t per_tile_t = (size_t)s->tiles * c.seq_len * SLAB_BYTES;
    int rc;
    if (c.module != DSP_SIGNAL_BILSTM) if ((rc = tc_alloc(m, (void**)&s->xseq_img, per_tile_t))) return rc;
    if (c.module != DSP_SEQ_BILSTM) if ((rc = tc_alloc(m, (void**)&s->xsig_img, per_tile_t))) return rc;
    if ((rc = tc_alloc(m, (void**)&s->ybuf[0], per_tile_t * 8))) return rc;
    if ((rc = tc_alloc(m, (void**)&s->ybuf[1], per_tile_t * 8))) return rc;
    if ((rc = tc_alloc(m, (void**)&s->comb_img, per_tile_t * 4))) return rc;
    if ((rc = tc_alloc(m, (void**)&s->hfinal, sizeof(float) * (size_t)s->tiles * TILE * 2 * c.hidden_size))) return rc;
    if ((rc = tc_alloc(m, (void**)&s->hfin_img, (size_t)s->tiles * 2 * (2 * c.hidden_size / 64) * SLAB_BYTES))) return rc;
    // activations of padding rows / the padding tile of an odd batch are read by the MMAs (results
    // discarded): keep them finite
    DSP_CUDA(cudaMemset(s->ybuf[0], 0, per_tile_t * 8));
    DSP_CUDA(cudaMemset(s->ybuf[1], 0, per_tile_t * 8));
    DSP_CUDA(cudaMemset(s->comb_img, 0, per_tile_t * 4));
    DSP_CUDA(cudaMemset(s->hfin_img, 0, (size_t)s->tiles * 2 * (2 * c.hidden_size / 64) * SLAB_BYTES));
    s->tc_head = c.num_classes <= HEAD_MAX_CLASSES;
    return DSP_OK;
}

bool tc_seq_split(const Model* m) {
    const TcState* s = (const TcState*)m->tc_state;
    return s && s->seq_split;
}

void tc_destroy(Model* m) {
    TcState* s = (TcState*)m->tc_state;
    if (!s) return;
    for (auto* p : s->lstm_packs) delete p;
    for (auto* p : s->dense_packs) delete p;
    delete s;
    m->tc_state = nullptr;
}

void tc_drop_packs(Model* m) {
    TcState* s = (TcState*)m->tc_state;
    if (!s) return;
    for (auto* p : s->lstm_packs) delete p;
    for (auto* p : s->dense_packs) delete p;
    s->lstm_packs.clear();
    s->dense_packs.clear();
    s->head_pack = nullptr;
}

int tc_pack_lstm_layer(Model* m, LstmLayer& L,
                       const float* wih0, const float* whh0, const float* bih0, const float* bhh0,
                       const float* wih1, const float* whh1, const float* bih1, const float* bhh1,
                       int split_first, int split_n, int len_col) {
    TcState* s = (TcState*)m->tc_state;
    const int H = L.H;
    int K = L.K;
    DSP_REQUIRE(H == 128 || H == 256, DSP_ERR_INVALID, "tcgen05 path: LSTM hidden size %d unsupported", H);
    // First layer of lstm_seq: the scalar features [split_first, split_first + split_n) arrive as FP16 value +
    // FP16 residual (prep_images_kernel), so their W_ih columns appear twice; the len column (and its twin) is
    // scaled by 1 / SEQ_LEN_SCALE.  Powers of two: the FP16 rounding of the weights is unchanged.
    std::vector<float> wext[2];
    if (split_n > 0) {
        const int K2 = K + split_n;
        const float* src[2] = {wih0, wih1};
        for (int d = 0; d < 2; ++d) {
            wext[d].assign((size_t)4 * H * K2, 0.f);
            for (int r = 0; r < 4 * H; ++r)
                for (int k = 0; k < K2; ++k) {
                    const int k0 = k < K ? k : split_first + (k - K);
                    wext[d][(size_t)r * K2 + k] = src[d][(size_t)r * K + k0] * (k0 == len_col ? 1.f / SEQ_LEN_SCALE : 1.f);
                }
        }
        wih0 = wext[0].data(); wih1 = wext[1].data();
        K = K2;
    }
    const int KSX = (K + 63) / 64, KSH = H / 64, KS = KSX + KSH, NCH = H / 32;
    DSP_REQUIRE(KSX == 1 || KSX == 4 || KSX == 8, DSP_ERR_INVALID, "tcgen05 path: LSTM input width %d unsupported", K);
    TcLstmPack* pk = new TcLstmPack();
    s->lstm_packs.push_back(pk);
    pk->KSX = KSX;
    pk->xk16 = (K + 15) / 16;
    const float* wih[2] = {wih0, wih1}; const float* whh[2] = {whh0, whh1};
    const float* bih[2] = {bih0, bih1}; const float* bhh[2] = {bhh0, bhh1};
    // branch_kernel / branch_fused_kernel stage BR_KSX x slabs per direction: the first layer of a branch, whose input
    // tc_create limits to 64 columns (signal_len <= 64, <= 16 sequence features), gets their weight image
    static_assert(BR_KSX == 1, "a branch's first-layer input is one slab wide");
    if (H == BR_H && KSX == BR_KSX) {
        // [rank][stream unit][32 rows x 128 B]; per chunk pair (c, c+1) the stream is
        // X(0,c) X(0,c+1) X(1,c) X(1,c+1) H(0,c) H(0,c+1) H(1,c) H(1,c+1) (first index = direction)
        std::vector<uint8_t> img((size_t)2 * BR_W_STEP * QSLAB_BYTES, 0);
        std::vector<float> bias((size_t)BR_NBIAS);
        auto put = [&](int rank, size_t unit, int row, int k, float v) {
            __half h = __float2half_rn(v);
            memcpy(&img[((size_t)rank * BR_W_STEP + unit) * QSLAB_BYTES + slab_offset_bytes((uint32_t)row, (uint32_t)k)], &h, 2);
        };
        for (int d = 0; d < 2; ++d)
            for (int ch = 0; ch < BR_NCH; ++ch) {
                const size_t pair_base = (size_t)(ch >> 1) * BR_PAIR_UNITS;
                const size_t sx = pair_base + (size_t)(d * 2 + (ch & 1)) * BR_KSX, sh = pair_base + 4 * BR_KSX + (size_t)(d * 2 + (ch & 1)) * BR_KSH;
                for (int n = 0; n < BR_NW; ++n) {
                    const int g = (n >> 1) & 3;
                    const int unit = ch * 16 + (n >> 3) * 2 + (n & 1);
                    const int wrow = g * H + unit;
                    const float scale = gate_scale(g);
                    bias[((size_t)d * BR_NCH + ch) * BR_NW + n] = scale * (bih[d][wrow] + bhh[d][wrow]);
                    for (int k = 0; k < K; ++k) put(n >> 5, sx + (k >> 6), n & 31, k & 63, scale * wih[d][(size_t)wrow * K + k]);
                    for (int k = 0; k < H; ++k) put(n >> 5, sh + (k >> 6), n & 31, k & 63, scale * whh[d][(size_t)wrow * H + k]);
                }
            }
        int rc;
        if ((rc = tc_alloc(m, (void**)&pk->w_img_dual, img.size()))) return rc;
        if ((rc = tc_alloc(m, (void**)&pk->bias_dual, bias.size() * sizeof(float)))) return rc;
        DSP_CUDA(cudaMemcpy(pk->w_img_dual, img.data(), img.size(), cudaMemcpyHostToDevice));
        DSP_CUDA(cudaMemcpy(pk->bias_dual, bias.data(), bias.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    const size_t per_rank = (size_t)NCH * KS;                       // half slabs per (dir, rank)
    std::vector<uint8_t> img((size_t)2 * 2 * per_rank * HSLAB_BYTES, 0);
    std::vector<float> bias((size_t)2 * NCH * 128);
    for (int d = 0; d < 2; ++d)
        for (int ch = 0; ch < NCH; ++ch) {
            // stream order of a chunk pair (c, c+1): X(c) X(c+1) H(c) H(c+1)
            const size_t pair_base = (size_t)(ch >> 1) * 2 * KS;
            const size_t sx = pair_base + (size_t)(ch & 1) * KSX, sh = pair_base + 2 * KSX + (size_t)(ch & 1) * KSH;
            for (int n = 0; n < 128; ++n) {
                // column n of the chunk: unit pair (n >> 3), gate (n >> 1) & 3, unit parity n & 1
                const int g = (n >> 1) & 3;
                const int unit = ch * 32 + (n >> 3) * 2 + (n & 1);
                const int wrow = g * H + unit;                      // torch gate blocks i,f,g,o
                // sigmoid(z) = 1/(1 + 2^(-log2e z)), tanh(z) = (1 - 2^(-2 log2e z))/(1 + 2^(-2 log2e z))
                const float scale = gate_scale(g);
                const size_t rank_base = ((size_t)d * 2 + (n >> 6)) * per_rank;
                bias[((size_t)d * NCH + ch) * 128 + n] = scale * (bih[d][wrow] + bhh[d][wrow]);
                for (int k = 0; k < K; ++k)
                    put_half(img, rank_base, sx + (k >> 6), n, k & 63, scale * wih[d][(size_t)wrow * K + k]);
                for (int k = 0; k < H; ++k)
                    put_half(img, rank_base, sh + (k >> 6), n, k & 63, scale * whh[d][(size_t)wrow * H + k]);
            }
        }
    int rc;
    if ((rc = tc_alloc(m, (void**)&pk->w_img, img.size()))) return rc;
    if ((rc = tc_alloc(m, (void**)&pk->bias, bias.size() * sizeof(float)))) return rc;
    DSP_CUDA(cudaMemcpy(pk->w_img, img.data(), img.size(), cudaMemcpyHostToDevice));
    DSP_CUDA(cudaMemcpy(pk->bias, bias.data(), bias.size() * sizeof(float), cudaMemcpyHostToDevice));
    L.tc = pk;
    return DSP_OK;
}

int tc_pack_dense(Model* m, DenseF32& D, const float* w, const float* b) {
    TcState* s = (TcState*)m->tc_state;
    // per-timestep fc layers and fc1 (K = 2J, J in {128, 256}) run on the tensor cores; fc2 is
    // applied in fp32 inside the head epilogue
    if (!(D.J == 128 || D.J == 256) || D.K != 2 * D.J) { D.tc = nullptr; return DSP_OK; }
    const int KS = D.K / 64, NCH = D.J / 128;
    TcDensePack* pk = new TcDensePack();
    s->dense_packs.push_back(pk);
    pk->KS = KS;
    const size_t per_rank = (size_t)NCH * KS;
    std::vector<uint8_t> img((size_t)2 * per_rank * HSLAB_BYTES, 0);
    for (int n = 0; n < D.J; ++n)
        for (int k = 0; k < D.K; ++k)
            put_half(img, (size_t)((n >> 6) & 1) * per_rank, (size_t)(n >> 7) * KS + (k >> 6), n & 127, k & 63, w[(size_t)n * D.K + k]);
    int rc;
    if ((rc = tc_alloc(m, (void**)&pk->w_img, img.size()))) return rc;
    if ((rc = tc_alloc(m, (void**)&pk->bias, sizeof(float) * D.J))) return rc;
    DSP_CUDA(cudaMemcpy(pk->w_img, img.data(), img.size(), cudaMemcpyHostToDevice));
    DSP_CUDA(cudaMemcpy(pk->bias, b, sizeof(float) * D.J, cudaMemcpyHostToDevice));
    D.tc = pk;
    return DSP_OK;
}

// fc1 for the head: three weight passes [W_hi, W_hi, W_lo] matching the activation passes
// [h_hi, h_lo, h_hi]: (h_hi + h_lo)(W_hi + W_lo) without the lo*lo term, i.e. fc1 to ~fp32 accuracy
// on the FP16 tensor pipe.
int tc_pack_head(Model* m, DenseF32& D, const float* w, const float* b) {
    TcState* s = (TcState*)m->tc_state;
    if (!(D.J == 256 && D.K == 512)) { s->tc_head = false; return DSP_OK; }
    const int KS = D.K / 64, NCH = D.J / 128;
    TcDensePack* pk = new TcDensePack();
    s->dense_packs.push_back(pk);
    s->head_pack = pk;
    pk->KS = KS;
    const size_t per_pass = (size_t)NCH * KS, per_rank = 3 * per_pass;
    std::vector<uint8_t> img((size_t)2 * per_rank * HSLAB_BYTES, 0);
    for (int n = 0; n < D.J; ++n)
        for (int k = 0; k < D.K; ++k) {
            const float wv = w[(size_t)n * D.K + k];
            const float hi = __half2float(__float2half_rn(wv));
            const size_t rank_base = (size_t)((n >> 6) & 1) * per_rank;
            const size_t slab = (size_t)(n >> 7) * KS + (k >> 6);
            put_half(img, rank_base, 0 * per_pass + slab, n & 127, k & 63, hi);
            put_half(img, rank_base, 1 * per_pass + slab, n & 127, k & 63, hi);
            put_half(img, rank_base, 2 * per_pass + slab, n & 127, k & 63, wv - hi);
        }
    int rc;
    if ((rc = tc_alloc(m, (void**)&pk->w_img, img.size()))) return rc;
    if ((rc = tc_alloc(m, (void**)&pk->bias, sizeof(float) * D.J))) return rc;
    DSP_CUDA(cudaMemcpy(pk->w_img, img.data(), img.size(), cudaMemcpyHostToDevice));
    DSP_CUDA(cudaMemcpy(pk->bias, b, sizeof(float) * D.J, cudaMemcpyHostToDevice));
    return DSP_OK;
}

int tc_forward_chunk(Model* m, const float* kmer, const float* means, const float* stds, const float* lens,
                     const float* signals, const float* const* h0, const float* const* c0,
                     const int64_t* sstride, uint64_t seed, uint64_t chunk_id, int64_t n,
                     float* logits, float* probs, int32_t* labels, cudaStream_t st) {
    TcState* s = (TcState*)m->tc_state;
    const dsp_config& c = m->cfg;
    const int T = c.seq_len, H = c.hidden_size;
    const int64_t tiles = ((n + TILE - 1) / TILE + 1) / 2 * 2;     // whole CTA pairs; padding rows are zero-filled
    const bool seq = c.module != DSP_SIGNAL_BILSTM, sig = c.module != DSP_SEQ_BILSTM;
    {
        Span sp(m, 0, st);
        const int64_t total = tiles * TILE * T;
        // Programmatic dependent launch here too: the images this kernel writes were last read by the first-layer
        // kernels of the PREVIOUS pass, which completed before that pass's head kernel could start its last wave, so
        // the feature assembly may fill the SMs the head kernel leaves idle while it drains.
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)((total + 255) / 256));
        cfg.blockDim = dim3(256);
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = s->pdl ? 1 : 0;
        DSP_CUDA(cudaLaunchKernelEx(&cfg, prep_images_kernel, kmer, means, stds, lens, signals, (const float*)m->embed,
                                    c.is_base ? c.embedding_size : 0, c.vocab_size, c.is_signallen, s->seq_split ? 1 : 0,
                                    c.signal_len, T, n, tiles * TILE, seq ? s->xseq_img : (uint8_t*)nullptr,
                                    sig ? s->xsig_img : (uint8_t*)nullptr));
        m->launches++;
    }
    auto run_stack = [&](std::vector<LstmLayer>& layers, const uint8_t* x0, int grp, int hid, bool is_comb) -> int {
        const uint8_t* x = x0;
        for (size_t l = 0; l < layers.size(); ++l) {
            TcLstmPack* pk = (TcLstmPack*)layers[l].tc;
            const bool final_layer = is_comb && l + 1 == layers.size();
            LayerParams p{};
            p.x_img = x; p.w_img = pk->w_img; p.bias = pk->bias;
            if (h0) {
                p.h0 = h0[grp] + (int64_t)l * 2 * sstride[grp]; p.c0 = c0[grp] + (int64_t)l * 2 * sstride[grp];
                p.state_dir_stride = sstride[grp];
            }
            p.seed = seed; p.rng_call = (uint32_t)chunk_id; p.rng_slot = (uint32_t)((grp * 8 + (int)l) * 2);
            p.site_base = (int64_t)chunk_id * m->cap;
            const bool head_tc = final_layer && s->tc_head;
            p.y_img = head_tc ? s->hfin_img : s->ybuf[l & 1]; p.hfinal = (final_layer && !head_tc) ? s->hfinal : nullptr;
            p.n = n; p.T = T; p.xk16 = pk->xk16; p.y_slabs = 2 * hid / 64; p.y_col_off = 0;
            p.write_y = final_layer ? (head_tc ? 2 : 0) : 1;
#ifdef DSP_MEAS_SKIP_Y
            // measurement BUILD only (DSP_B200_VARIANT=skipy DSP_B200_DEFINES=-DDSP_MEAS_SKIP_Y, bench.py --meas-skip-y):
            // skip the inter-layer activation stores of the hidden-256 layers once the images hold realistic data
            // from earlier passes, to price those stores.  Results are wrong; the shipped library has no such switch.
            if (p.write_y == 1 && hid == 256) { const char* e = getenv("DSP_B200_SKIP_Y_NOW"); if (e && atoi(e)) p.write_y = 0; }
#endif
            Span sp(m, is_comb ? 1 : 4, st);
            // Two ways to run a hidden-128 layer: one CTA pair per (tile pair, direction), or both directions
            // as two chains of one CTA pair (branch_kernel: ~1.8x the time per CTA for 2x the work).  Pick
            // by whole waves: 2 x tiles CTAs of cost 1 against tiles CTAs of cost 1.8.
            bool dual = pk->w_img_dual != nullptr;
            if (dual) {
                const int64_t sms = m->n_sm > 0 ? m->n_sm : 148;
                const double single_cost = (double)((2 * tiles + sms - 1) / sms);
                const double dual_cost = 1.8 * (double)((tiles + sms - 1) / sms);
                dual = dual_cost < single_cost;
                if (s->force_dual >= 0) dual = s->force_dual != 0;
            }
            if (dual) { p.w_img = pk->w_img_dual; p.bias = pk->bias_dual; }
            int rc = dual ? launch_branch(m, p, tiles, st) : launch_lstm(m, pk->KSX, hid, p, tiles, st);
            if (rc) return rc;
            x = s->ybuf[l & 1];
        }
        return DSP_OK;
    };
    auto run_fc = [&](DenseF32& D, const uint8_t* x, int col_off) -> int {
        TcDensePack* pk = (TcDensePack*)D.tc;
        DSP_REQUIRE(pk != nullptr, DSP_ERR_INVALID, "tcgen05 path: dense layer %dx%d unsupported", D.J, D.K);
        LayerParams p{};
        p.x_img = x; p.w_img = pk->w_img; p.bias = pk->bias; p.y_img = s->comb_img; p.n = n; p.T = T;
        p.xk16 = pk->KS * 4; p.y_slabs = H / 64; p.y_col_off = col_off; p.write_y = 1;
        Span sp(m, 2, st);
        return launch_fc(m, pk->KS, D.J, p, tiles, st);
    };
    int rc;
    int comb_off = 0;
    // both_bilstm with one-layer hidden-128 branches (the shipped configuration): both branches and their fc
    // layers as ONE launch (branch_fused_kernel).  DSP_B200_BRANCH_DUAL=0|1 (read at handle creation) keeps the
    // separate launches for A/B measurements and for the tests that cover those kernels.
    bool fused = seq && sig && s->force_dual < 0 && m->lstm_seq.size() == 1 && m->lstm_signal.size() == 1 &&
                 m->nhid_seq == BR_H && m->nhid_signal == BR_H && H == 256;
    if (fused) {
        TcLstmPack* pk[2] = {(TcLstmPack*)m->lstm_seq[0].tc, (TcLstmPack*)m->lstm_signal[0].tc};
        TcDensePack* fk[2] = {(TcDensePack*)m->fc_seq.tc, (TcDensePack*)m->fc_signal.tc};
        fused = pk[0] && pk[1] && fk[0] && fk[1] && pk[0]->w_img_dual && pk[1]->w_img_dual && pk[0]->KSX == 1 && pk[1]->KSX == 1 &&
                fk[0]->KS == 4 && fk[1]->KS == 4;
        if (fused) {
            FusedBranchParams p{};
            const uint8_t* ximg[2] = {s->xseq_img, s->xsig_img};
            for (int b = 0; b < 2; ++b) {
                p.x_img[b] = ximg[b]; p.w_img[b] = pk[b]->w_img_dual; p.bias[b] = pk[b]->bias_dual;
                if (h0) { p.h0[b] = h0[b]; p.c0[b] = c0[b]; p.state_dir_stride[b] = sstride[b]; }
                p.rng_slot[b] = (uint32_t)((b * 8) * 2);
                p.xk16[b] = pk[b]->xk16;
                p.y_img[b] = s->ybuf[b];
                p.fcw_img[b] = fk[b]->w_img; p.fcb[b] = fk[b]->bias;
            }
            p.comb_img = s->comb_img; p.seed = seed; p.rng_call = (uint32_t)chunk_id; p.site_base = (int64_t)chunk_id * m->cap;
            p.n = n; p.T = T;
            Span sp(m, 4, st);
            if ((rc = launch_branch_fused(m, p, tiles, st))) return rc;
        }
    }
    if (fused) {
        // nothing left to do before lstm_comb
    } else if (seq) {
        if ((rc = run_stack(m->lstm_seq, s->xseq_img, 0, m->nhid_seq, false))) return rc;
        if ((rc = run_fc(m->fc_seq, s->ybuf[(m->lstm_seq.size() - 1) & 1], 0))) return rc;
        comb_off = m->nhid_seq;
    }
    if (!fused && sig) {
        if ((rc = run_stack(m->lstm_signal, s->xsig_img, 1, m->nhid_signal, false))) return rc;
        if ((rc = run_fc(m->fc_signal, s->ybuf[(m->lstm_signal.size() - 1) & 1], comb_off))) return rc;
    }
    if ((rc = run_stack(m->lstm_comb, s->comb_img, 2, H, true))) return rc;
    Span sp(m, 3, st);
    if (!s->tc_head) return f32_head_flat(m, s->hfinal, n, logits, probs, labels, st);
    TcDensePack* pk = s->head_pack;
    DSP_REQUIRE(pk != nullptr && pk->KS == 8 && m->fc1.J == 256, DSP_ERR_INVALID, "tcgen05 path: head shape unsupported");
    LayerParams p{};
    p.x_img = s->hfin_img; p.w_img = pk->w_img; p.bias = pk->bias; p.n = n; p.T = 3; p.xk16 = 32;
    p.w2t = m->fc2.wt; p.b2 = m->fc2.bias; p.logits = logits; p.probs = probs; p.labels = labels; p.num_classes = c.num_classes;
    return launch_layer<8, 0, MODE_HEAD, 256>(m, p, tiles, st);
}

}  // namespace dsp
