// Multi-GPU call_freq: the one exchange step of the path (SURVEY.md 8(e)), as kernels over NVLink
// peer memory instead of a library all-to-all.  The same windows also carry the deterministic gradient
// all-reduce of multi-GPU training (dsp_comm_allreduce_f32, below the splitters).
//
// One process per GPU.  Every rank owns two receive WINDOWS and a small control block in device
// memory, exported to the other ranks of the box with CUDA IPC (dsp_comm_export / _connect), so a
// kernel on GPU s can store straight into GPU d's HBM through NVLink 5 / NVSwitch.  An exchange is
// then the stable partition of route.cuh whose scatter kernel writes each item at its FINAL position
// in the destination's window -- partition and all-to-all are one pass, there is no send buffer, no
// host-side split-size bookkeeping and no NCCL call:
//
//   count (per block, per destination)  ->  scan  ->  publish my counts row into every
//   peer's control block, then a release flag  ->  prepare: wait for every rank's row, derive the
//   write bases (segments in source-rank order = global file order) and check window capacity  ->
//   scatter over NVLink  ->  signal "my stores have landed" to every peer, wait for everybody's signal.
//
// All of it is stream ordered; the host synchronises once per exchange to learn the receive count.
// Records of one site all go to hash(key) % world, arrive grouped by source rank in file order, and
// are aggregated by the same sort + ordered replay as on one GPU (freq.cu): the float64 sums are the
// reference's bit for bit (no partial-sum merging -- float64 addition is order sensitive,
// call_mods_freq.py:60-61).  Site rows then travel to the rank that parsed their first callable
// record (which holds strand / pos_in_strand / k-mer, :55-59) with the same machinery.
#include "freq.cuh"
#include "route.cuh"
#include <unistd.h>
#include <algorithm>
#include <cstring>
#include <vector>

namespace dsp {

int sort_rows(Scratch& sc, cudaStream_t st, const SiteRow* rows, int64_t n, int by_key, SiteRow* out, int end_bit);

namespace {

using route::MAXW;

struct Ctrl {                                   // device memory; peers write, the owner reads
    int64_t cnt[2][MAXW][MAXW];                 // [epoch parity][source][destination]
    unsigned long long bits[2][MAXW];           // OR of the keys a source routes
    unsigned long long flag_cnt[MAXW];          // epoch of source's last count publication
    unsigned long long flag_data[MAXW];         // epoch of source's last "stores landed" signal
    uint64_t samples[2][MAXW][256];             // splitter selection: every rank's sample of its rows' sort field
    int32_t nsamples[2][MAXW];
    unsigned long long flag_smp[MAXW];
    unsigned long long flag_ar[2][MAXW];         // all-reduce: [0] slots of source landed here, [1] its summed range landed here
};
constexpr int NSAMP = 256;

struct Result { int64_t n_recv; unsigned long long bits; int32_t err; int32_t pad; };   // err: 1 window overflow, 2 peer timeout

struct Peers { Ctrl* ctrl[MAXW]; };

struct Blob {                                   // what dsp_comm_export hands to the other ranks
    int64_t pid; int32_t device, rank; uint64_t ptr[3];
    cudaIpcMemHandle_t h[3];
};

constexpr unsigned long long SPIN_TIMEOUT_NS = 30ull * 1000 * 1000 * 1000;

__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// spin until *flag >= epoch (written by a peer GPU through NVLink); false on timeout
__device__ __forceinline__ bool wait_flag(const unsigned long long* flag, unsigned long long epoch) {
    const unsigned long long t0 = gtime();
    while (*reinterpret_cast<const volatile unsigned long long*>(flag) < epoch) {
        if (gtime() - t0 > SPIN_TIMEOUT_NS) return false;
        __nanosleep(200);
    }
    return true;
}

__global__ void publish_kernel(const int64_t* __restrict__ totals, Peers peers, int me, int world, int parity, unsigned long long epoch) {
    const int t = threadIdx.x;
    if (t < world * world) { const int p = t / world, d = t % world; peers.ctrl[p]->cnt[parity][me][d] = totals[d]; }
    __threadfence_system();
    __syncthreads();
    if (t < world) *reinterpret_cast<volatile unsigned long long*>(&peers.ctrl[t]->flag_cnt[me]) = epoch;
}

struct Windows { void* win[MAXW]; };

__global__ void prepare_kernel(const Ctrl* __restrict__ local, Windows wins, int me, int world, int parity,
                               unsigned long long epoch, int64_t cap_items, route::Targets* __restrict__ tg,
                               int* __restrict__ abort_flag, Result* __restrict__ res) {
    __shared__ int s_bad;
    const int t = threadIdx.x;
    if (t == 0) s_bad = 0;
    __syncthreads();
    if (t < world && !wait_flag(&local->flag_cnt[t], epoch)) atomicOr(&s_bad, 2);
    __threadfence_system();
    __syncthreads();
    if (t < world) {
        int64_t base = 0, tot = 0;
        for (int s = 0; s < world; ++s) {
            const int64_t c = local->cnt[parity][s][t];
            if (s < me) base += c;
            tot += c;
        }
        tg->dst[t] = wins.win[t];
        tg->base[t] = base;
        if (tot > cap_items) atomicOr(&s_bad, 1);
        if (t == me) res->n_recv = tot;
    }
    __syncthreads();
    if (t == 0) {
        res->err = s_bad;
        *abort_flag = s_bad;
    }
}

// `key_bits`: OR of the keys this rank's scatter wrote (to anybody); every receiver ORs what its sources report, a
// superset of the bits of the keys it holds -- all the squeeze of the sort key needs.
__global__ void signal_wait_kernel(Ctrl* local, Peers peers, int me, int world, int parity, unsigned long long epoch,
                                   const unsigned long long* __restrict__ key_bits, Result* __restrict__ res) {
    const int t = threadIdx.x;
    if (t < world) peers.ctrl[t]->bits[parity][me] = *key_bits;
    __threadfence_system();                      // the scatter kernel's peer stores (previous kernel of the stream) before the flag
    if (t < world) *reinterpret_cast<volatile unsigned long long*>(&peers.ctrl[t]->flag_data[me]) = epoch;
    bool ok = true;
    if (t < world) ok = wait_flag(&local->flag_data[t], epoch);
    __threadfence_system();
    unsigned long long b = (t < world && ok) ? *reinterpret_cast<const volatile unsigned long long*>(&local->bits[parity][t]) : 0ull;
    const unsigned blo = __reduce_or_sync(0xffffffffu, (unsigned)b), bhi = __reduce_or_sync(0xffffffffu, (unsigned)(b >> 32));
    if (t == 0) res->bits = ((unsigned long long)bhi << 32) | blo;
    if (!ok) atomicOr(&res->err, 2);
}

// ---- balanced row placement: splitters of the `first` field chosen from every rank's sample ---------------------
// Sites are spread over the ranks by key hash, but their FIRST callable records are not: with reads in random order
// nearly every site is first seen in rank 0's shard, so sending rows to the rank that parsed that record would funnel
// the whole table through one GPU.  Instead every rank publishes NSAMP evenly spaced `first` values of its rows to
// all peers, everybody sorts the same world x NSAMP values and cuts them into `world` equal parts: the rows then go to
// the rank whose [bounds[r], bounds[r+1]) holds their `first`, sorted there -- the slices of ranks 0..world-1 still
// concatenate to dict insertion order, and every rank holds about 1/world of the table.
__global__ void publish_samples_kernel(const SiteRow* __restrict__ rows, int64_t n, Peers peers, int me, int world, int parity,
                                       unsigned long long epoch) {
    const int t = threadIdx.x;                                 // NSAMP threads
    const int ns = (int)(n < NSAMP ? n : NSAMP);
    if (t < ns) {
        const uint64_t v = rows[(int64_t)(((double)t + 0.5) * (double)n / (double)ns)].first;
        for (int p = 0; p < world; ++p) peers.ctrl[p]->samples[parity][me][t] = v;
    }
    if (t < world) peers.ctrl[t]->nsamples[parity][me] = ns;
    __threadfence_system();
    __syncthreads();
    if (t < world) *reinterpret_cast<volatile unsigned long long*>(&peers.ctrl[t]->flag_smp[me]) = epoch;
}

__global__ void __launch_bounds__(1024) splitters_kernel(const Ctrl* local, int world, int parity, unsigned long long epoch,
                                                         uint64_t* __restrict__ bounds, Result* __restrict__ res) {
    __shared__ uint64_t s[MAXW * NSAMP];
    __shared__ int s_n, s_bad;
    const int t = threadIdx.x;
    if (t == 0) { s_n = 0; s_bad = 0; }
    __syncthreads();
    if (t < world && !wait_flag(&local->flag_smp[t], epoch)) atomicOr(&s_bad, 2);
    __threadfence_system();
    __syncthreads();
    for (int i = t; i < MAXW * NSAMP; i += 1024) {
        const int r = i / NSAMP, j = i % NSAMP;
        const bool ok = r < world && j < *reinterpret_cast<const volatile int32_t*>(&local->nsamples[parity][r]);
        s[i] = ok ? *reinterpret_cast<const volatile uint64_t*>(&local->samples[parity][r][j]) : ~0ull;
        if (ok) atomicAdd(&s_n, 1);
    }
    __syncthreads();
    for (int k = 2; k <= MAXW * NSAMP; k <<= 1)                 // bitonic sort, ascending; the padding sorts last
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = t; i < MAXW * NSAMP; i += 1024) {
                const int l = i ^ j;
                if (l > i) {
                    const uint64_t a = s[i], b = s[l];
                    if (((i & k) == 0) ? (a > b) : (a < b)) { s[i] = b; s[l] = a; }
                }
            }
            __syncthreads();
        }
    if (t <= world) {
        uint64_t v = t == 0 ? 0ull : ~0ull;
        if (t > 0 && t < world && s_n > 0) v = s[(int)(((int64_t)s_n * t) / world)];
        bounds[t] = v;
    }
    if (t == 0 && s_bad) res->err = s_bad;
}

// ---- deterministic fp32 all-reduce of a tensor list (dsp_comm_allreduce_f32) -------------------------------------
// The list is one flat vector of E floats, the tensors back to back in argument order.  Rank r owns the range
// [r * chunk, min(E, (r + 1) * chunk)), chunk = ceil(E / world) rounded up to a multiple of 4 (16-byte aligned).
//   pack:          every rank stores the part of its vector that rank r owns into slot [me] of r's window 0
//   signal + wait  on flag_ar[0]
//   reduce:        the owner adds its world slots in rank order, fl(fl(s0 + s1) + s2)..., and stores the sums into
//                  every rank's window 1 at the range's offset
//   signal + wait  on flag_ar[1]
//   unpack:        window 1 -> the tensors
// One rank computes each element, with plain adds in a fixed order, so every rank gets the same bits on every call,
// whatever the chunking and timing.  The kernels that move data never spin; only the one-warp signal kernels wait,
// so ranks that share a GPU make progress under time-slicing.
//
// No window is overwritten while a peer may still read it:
// * slot writes of call k+1 into owner r's window 0, against r's reduction of call k: a rank packs call k+1 only after
//   its call-k wait on flag_ar[1] saw every rank's flag, and r raises that flag in the kernel after its reduction, so
//   r has finished reading window 0 for call k.
// * window-1 writes of call k+1 by owner r into rank p's window 1, against p's unpack of call k: r reduces call k+1
//   only after its wait on flag_ar[0] saw p's flag of call k+1, which p raises after its pack of call k+1, and p's
//   stream runs that pack after its unpack of call k.
constexpr int AR_MAXT = 64;                     // tensors per pack / unpack launch (kernel parameter space)
constexpr int AR_THREADS = 256;

struct ArList {
    float* ptr[AR_MAXT];
    int64_t off[AR_MAXT + 1];                   // flat offsets of the tensors; off[count] = end of the group
    int count;
};

__host__ __device__ __forceinline__ int64_t ar_chunk(int64_t e, int world) { return ((e + world - 1) / world + 3) & ~(int64_t)3; }

// the tensor that holds flat index j: the last one starting at or before j (empty tensors share their successor's start)
__device__ __forceinline__ int ar_find(const int64_t* off, int count, int64_t j) {
    int lo = 0, hi = count - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= j) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(AR_THREADS) allreduce_pack_kernel(ArList l, Windows win0, int me, int64_t chunk) {
    __shared__ float* s_ptr[AR_MAXT];
    __shared__ int64_t s_off[AR_MAXT + 1];
    __shared__ float* s_win[MAXW];               // tables indexed at run time: shared memory, not a stack copy of the parameters
    for (int i = threadIdx.x; i <= l.count; i += AR_THREADS) {
        s_off[i] = l.off[i];
        if (i < l.count) s_ptr[i] = l.ptr[i];
    }
    if (threadIdx.x == 0) {
#pragma unroll
        for (int r = 0; r < MAXW; ++r) s_win[r] = static_cast<float*>(win0.win[r]);
    }
    __syncthreads();
    const int64_t base = s_off[0], n = s_off[l.count] - base;
    for (int64_t i = (int64_t)blockIdx.x * AR_THREADS + threadIdx.x; i < n; i += (int64_t)gridDim.x * AR_THREADS) {
        const int64_t j = base + i;
        const int t = ar_find(s_off, l.count, j);
        const float v = s_ptr[t][j - s_off[t]];
        const int64_t r = j / chunk;
        s_win[r][me * chunk + (j - r * chunk)] = v;
    }
}

__global__ void __launch_bounds__(AR_THREADS) allreduce_reduce_kernel(const float* __restrict__ slots, Windows win1, int world,
                                                                      int64_t chunk, int64_t lo, int64_t len,
                                                                      const int* __restrict__ abort_flag) {
    __shared__ float* s_win[MAXW];
    if (*abort_flag) return;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int r = 0; r < MAXW; ++r) s_win[r] = static_cast<float*>(win1.win[r]);
    }
    __syncthreads();
    const int64_t nv = len >> 2, stride = (int64_t)gridDim.x * AR_THREADS;
    for (int64_t v = (int64_t)blockIdx.x * AR_THREADS + threadIdx.x; v < nv; v += stride) {
        float4 a = reinterpret_cast<const float4*>(slots)[v];
        for (int s = 1; s < world; ++s) {
            const float4 b = reinterpret_cast<const float4*>(slots + s * chunk)[v];
            a.x = __fadd_rn(a.x, b.x); a.y = __fadd_rn(a.y, b.y); a.z = __fadd_rn(a.z, b.z); a.w = __fadd_rn(a.w, b.w);
        }
        for (int p = 0; p < world; ++p) reinterpret_cast<float4*>(s_win[p] + lo)[v] = a;
    }
    if (blockIdx.x == 0 && threadIdx.x < (len & 3)) {                  // the last range may end off a multiple of 4
        const int64_t i = (nv << 2) + threadIdx.x;
        float a = slots[i];
        for (int s = 1; s < world; ++s) a = __fadd_rn(a, slots[s * chunk + i]);
        for (int p = 0; p < world; ++p) s_win[p][lo + i] = a;
    }
}

__global__ void __launch_bounds__(AR_THREADS) allreduce_unpack_kernel(ArList l, const float* __restrict__ win1,
                                                                      const int* __restrict__ abort_flag) {
    __shared__ float* s_ptr[AR_MAXT];
    __shared__ int64_t s_off[AR_MAXT + 1];
    if (*abort_flag) return;
    for (int i = threadIdx.x; i <= l.count; i += AR_THREADS) {
        s_off[i] = l.off[i];
        if (i < l.count) s_ptr[i] = l.ptr[i];
    }
    __syncthreads();
    const int64_t base = s_off[0], n = s_off[l.count] - base;
    for (int64_t i = (int64_t)blockIdx.x * AR_THREADS + threadIdx.x; i < n; i += (int64_t)gridDim.x * AR_THREADS) {
        const int64_t j = base + i;
        const int t = ar_find(s_off, l.count, j);
        s_ptr[t][j - s_off[t]] = win1[j];
    }
}

// One warp: "my stores of this phase have landed" to every peer, then wait for every peer's.  After a time-out the
// rank raises no further flag, so its peers time out too instead of unpacking a range that was never summed.
__global__ void allreduce_signal_wait_kernel(Ctrl* local, Peers peers, int me, int world, int phase, unsigned long long epoch,
                                             int* abort_flag, Result* res) {
    const int t = threadIdx.x;
    if (*reinterpret_cast<volatile int*>(abort_flag)) return;
    __threadfence_system();                      // the previous kernel's peer stores before the flag
    if (t < world) *reinterpret_cast<volatile unsigned long long*>(&peers.ctrl[t]->flag_ar[phase][me]) = epoch;
    const bool ok = t >= world || wait_flag(&local->flag_ar[phase][t], epoch);
    __threadfence_system();
    if (!__all_sync(0xffffffffu, ok) && t == 0) {
        res->err |= 2;
        *abort_flag = 1;
    }
}

}  // namespace
}  // namespace dsp

struct dsp_comm_s {
    int device = 0, rank = 0, world = 1;
    int64_t window_bytes = 0;
    void* win[2] = {nullptr, nullptr};
    dsp::Ctrl* ctrl = nullptr;
    void* peer_win[2][dsp::route::MAXW] = {};
    dsp::Ctrl* peer_ctrl[dsp::route::MAXW] = {};
    bool opened[3][dsp::route::MAXW] = {};
    bool connected = false;
    unsigned long long epoch = 0;                // one per collective operation; the flags carry it
    unsigned long long n_exchanges = 0, n_samplings = 0;   // their parities pick the half of the count matrix / sample table
    dsp::route::Targets* d_tg = nullptr;
    int* d_abort = nullptr;
    dsp::Result* d_res = nullptr;
    dsp::Result* h_res = nullptr;                // pinned
    uint64_t* d_bounds = nullptr;                // world + 1 range bounds of the current row exchange
    uint64_t* h_bounds = nullptr;                // pinned
    int n_sm = 148;
    float last_ms[4] = {0, 0, 0, 0};             // route records, aggregate, route rows, order (CUDA events of the last call)
    cudaEvent_t ev[5] = {};
    // inside an exchange (window 0 = records, 1 = rows): count+scan+publish | wait for every rank's counts | scatter |
    // signal + wait for every rank's stores
    float detail_ms[2][4] = {};
    cudaEvent_t dev[2][5] = {};
};

using namespace dsp;

namespace {

struct DevGuard {
    int prev = -1;
    explicit DevGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// One exchange: items of `src` -> window `which` of their destination rank.  *n_recv / *bits: what this rank
// received.  Synchronises `st`.
template <typename Src>
int exchange(dsp_comm_s* c, Scratch& sc, cudaStream_t st, const Src& src, int64_t n, int which, size_t item_bytes,
             int64_t* n_recv, unsigned long long* bits) {
    using namespace route;
    DSP_REQUIRE(c->connected, DSP_ERR_STATE, "dsp_comm: not connected (dsp_comm_connect after exchanging the export blobs)");
    const Plan plan = make_plan(n, c->n_sm);
    int32_t* blk_counts; int64_t* blk_off; int64_t* totals; unsigned long long* d_bits;
    int rc;
    if ((rc = sc.alloc(&blk_counts, (size_t)plan.blocks * MAXD)) || (rc = sc.alloc(&blk_off, (size_t)plan.blocks * MAXD)) ||
        (rc = sc.alloc(&totals, MAXD)) || (rc = sc.alloc(&d_bits, 1))) return rc;
    // consecutive exchanges alternate between the two halves of the count matrix: a rank that runs ahead publishes the
    // next exchange's counts while a slower peer may still be reading this one's
    const unsigned long long epoch = ++c->epoch;
    const int parity = (int)(++c->n_exchanges & 1);
    Peers peers{}; Windows wins{};
    for (int r = 0; r < c->world; ++r) { peers.ctrl[r] = c->peer_ctrl[r]; wins.win[r] = c->peer_win[which][r]; }
    cudaEvent_t* ev = c->dev[which];
    DSP_CUDA(cudaMemsetAsync(d_bits, 0, sizeof(unsigned long long), st));
    cudaEventRecord(ev[0], st);
    count_kernel<Src><<<plan.blocks, RT, 0, st>>>(src, plan, c->world, blk_counts);
    scan_kernel<<<1, MAXD * 32, 0, st>>>(blk_counts, plan.blocks, c->world, blk_off, totals);
    publish_kernel<<<1, 256, 0, st>>>(totals, peers, c->rank, c->world, parity, epoch);
    cudaEventRecord(ev[1], st);
    prepare_kernel<<<1, 32, 0, st>>>(c->ctrl, wins, c->rank, c->world, parity, epoch, (int64_t)(c->window_bytes / item_bytes),
                                     c->d_tg, c->d_abort, c->d_res);
    cudaEventRecord(ev[2], st);
    ScatterLaunch<Src>::run(src, plan, c->world, blk_off, c->d_tg, c->d_abort, d_bits, st);
    cudaEventRecord(ev[3], st);
    signal_wait_kernel<<<1, 32, 0, st>>>(c->ctrl, peers, c->rank, c->world, parity, epoch, d_bits, c->d_res);
    cudaEventRecord(ev[4], st);
    DSP_CUDA(cudaGetLastError());
    DSP_CUDA(cudaMemcpyAsync(c->h_res, c->d_res, sizeof(Result), cudaMemcpyDeviceToHost, st));
    DSP_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < 4; ++i) cudaEventElapsedTime(&c->detail_ms[which][i], ev[i], ev[i + 1]);
    DSP_REQUIRE(!(c->h_res->err & 2), DSP_ERR_CUDA, "dsp_comm: rank %d timed out waiting for a peer (exchange %llu)", c->rank, epoch);
    DSP_REQUIRE(!(c->h_res->err & 1), DSP_ERR_NOMEM,
                "dsp_comm: a receive window (%lld items of %zu bytes) would overflow; create the communicator with larger windows",
                (long long)(c->window_bytes / item_bytes), item_bytes);
    *n_recv = c->h_res->n_recv;
    if (bits) *bits = c->h_res->bits;
    return DSP_OK;
}

// bounds_host != nullptr: upload them; nullptr: c->d_bounds already holds the bounds (splitters_kernel)
template <int UNITS>
int route_rows_units(dsp_comm_s* c, Scratch& sc, cudaStream_t st, const void* rows, int64_t n, int field_word,
                     const uint64_t* bounds_host, int64_t* n_recv) {
    typedef route::RowsByRange<UNITS> Src;
    if (bounds_host) {
        for (int w = 0; w <= c->world; ++w) c->h_bounds[w] = bounds_host[w];
        DSP_CUDA(cudaMemcpyAsync(c->d_bounds, c->h_bounds, sizeof(uint64_t) * (c->world + 1), cudaMemcpyHostToDevice, st));
    }
    Src src{};
    src.rows = reinterpret_cast<const typename Src::Item*>(rows);
    src.field_word = field_word;
    src.world = c->world;
    src.bounds = c->d_bounds;
    return exchange<Src>(c, sc, st, src, n, 1, (size_t)UNITS * 16, n_recv, nullptr);
}

// choose c->d_bounds so that the `first` fields of all ranks' rows fall into `world` equal parts
int choose_row_splitters(dsp_comm_s* c, cudaStream_t st, const SiteRow* rows, int64_t n) {
    const unsigned long long epoch = ++c->epoch;
    const int parity = (int)(++c->n_samplings & 1);
    Peers peers{};
    for (int r = 0; r < c->world; ++r) peers.ctrl[r] = c->peer_ctrl[r];
    publish_samples_kernel<<<1, NSAMP, 0, st>>>(rows, n, peers, c->rank, c->world, parity, epoch);
    splitters_kernel<<<1, 1024, 0, st>>>(c->ctrl, c->world, parity, epoch, c->d_bounds, c->d_res);
    DSP_CUDA(cudaGetLastError());
    return DSP_OK;
}

}  // namespace

extern "C" {

int dsp_comm_create(dsp_comm* out, int device, int rank, int world, int64_t window_bytes) {
    DSP_REQUIRE(out, DSP_ERR_INVALID, "dsp_comm_create: null argument");
    *out = nullptr;
    DSP_REQUIRE(world >= 1 && world <= route::MAXW && rank >= 0 && rank < world, DSP_ERR_INVALID,
                "dsp_comm_create: rank %d of %d (at most %d ranks: the GPUs of one box)", rank, world, route::MAXW);
    DSP_REQUIRE(window_bytes >= 4096, DSP_ERR_INVALID, "dsp_comm_create: window_bytes too small");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("dsp_comm_create: no CUDA device available; this library has no CPU path");
        return DSP_ERR_CUDA;
    }
    DSP_REQUIRE(device >= 0 && device < ndev, DSP_ERR_INVALID, "dsp_comm_create: bad device %d", device);
    DevGuard g(device);
    dsp_comm_s* c = new dsp_comm_s();
    c->device = device; c->rank = rank; c->world = world;
    c->window_bytes = (window_bytes + 255) & ~(int64_t)255;
    cudaDeviceGetAttribute(&c->n_sm, cudaDevAttrMultiProcessorCount, device);
    cudaError_t e = cudaSuccess;
    for (int w = 0; w < 2 && e == cudaSuccess; ++w) e = cudaMalloc(&c->win[w], (size_t)c->window_bytes);
    if (e == cudaSuccess) e = cudaMalloc((void**)&c->ctrl, sizeof(Ctrl));
    if (e == cudaSuccess) e = cudaMemset(c->ctrl, 0, sizeof(Ctrl));
    if (e == cudaSuccess) e = cudaMalloc((void**)&c->d_tg, sizeof(route::Targets));
    if (e == cudaSuccess) e = cudaMalloc((void**)&c->d_abort, sizeof(int));
    if (e == cudaSuccess) e = cudaMalloc((void**)&c->d_res, sizeof(Result));
    if (e == cudaSuccess) e = cudaMemset(c->d_res, 0, sizeof(Result));
    if (e == cudaSuccess) e = cudaMallocHost((void**)&c->h_res, sizeof(Result));
    if (e == cudaSuccess) e = cudaMalloc((void**)&c->d_bounds, sizeof(uint64_t) * (route::MAXW + 1));
    if (e == cudaSuccess) e = cudaMallocHost((void**)&c->h_bounds, sizeof(uint64_t) * (route::MAXW + 1));
    for (int i = 0; i < 5 && e == cudaSuccess; ++i) e = cudaEventCreate(&c->ev[i]);
    for (int i = 0; i < 10 && e == cudaSuccess; ++i) e = cudaEventCreate(&c->dev[i / 5][i % 5]);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        set_error("dsp_comm_create: %s (two windows of %lld bytes)", cudaGetErrorString(e), (long long)c->window_bytes);
        dsp_comm_destroy(c);
        return e == cudaErrorMemoryAllocation ? DSP_ERR_NOMEM : DSP_ERR_CUDA;
    }
    c->peer_win[0][rank] = c->win[0]; c->peer_win[1][rank] = c->win[1]; c->peer_ctrl[rank] = c->ctrl;
    c->connected = world == 1;
    *out = c;
    return DSP_OK;
}

int dsp_comm_export(dsp_comm c, void* blob, int64_t blob_cap, int64_t* blob_bytes) {
    DSP_REQUIRE(c && blob_bytes, DSP_ERR_INVALID, "dsp_comm_export: null argument");
    *blob_bytes = (int64_t)sizeof(Blob);
    DSP_REQUIRE(blob && blob_cap >= (int64_t)sizeof(Blob), DSP_ERR_NOMEM, "dsp_comm_export: blob needs %zu bytes", sizeof(Blob));
    DevGuard g(c->device);
    Blob b;
    memset(&b, 0, sizeof(b));
    b.pid = (int64_t)getpid(); b.device = c->device; b.rank = c->rank;
    void* ptrs[3] = {c->win[0], c->win[1], c->ctrl};
    for (int i = 0; i < 3; ++i) {
        b.ptr[i] = (uint64_t)(uintptr_t)ptrs[i];
        DSP_CUDA(cudaIpcGetMemHandle(&b.h[i], ptrs[i]));
    }
    memcpy(blob, &b, sizeof(b));
    return DSP_OK;
}

int dsp_comm_connect(dsp_comm c, const void* blobs, int64_t blob_bytes) {
    DSP_REQUIRE(c && blobs, DSP_ERR_INVALID, "dsp_comm_connect: null argument");
    DSP_REQUIRE(blob_bytes == (int64_t)sizeof(Blob), DSP_ERR_INVALID, "dsp_comm_connect: blob size %lld, expected %zu",
                (long long)blob_bytes, sizeof(Blob));
    DevGuard g(c->device);
    for (int r = 0; r < c->world; ++r) {
        if (r == c->rank) continue;
        Blob b;
        memcpy(&b, (const char*)blobs + (size_t)r * sizeof(Blob), sizeof(b));
        DSP_REQUIRE(b.rank == r, DSP_ERR_INVALID, "dsp_comm_connect: blob %d comes from rank %d (gather them in rank order)", r, b.rank);
        void* ptrs[3] = {nullptr, nullptr, nullptr};
        if (b.pid == (int64_t)getpid()) {          // ranks as threads of one process (tests): plain pointers, peer access on
            if (b.device != c->device) {
                cudaError_t e = cudaDeviceEnablePeerAccess(b.device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
                    set_error("dsp_comm_connect: no peer access %d -> %d: %s", c->device, b.device, cudaGetErrorString(e));
                    return DSP_ERR_CUDA;
                }
                cudaGetLastError();
            }
            for (int i = 0; i < 3; ++i) ptrs[i] = (void*)(uintptr_t)b.ptr[i];
        } else {
            for (int i = 0; i < 3; ++i) {
                cudaError_t e = cudaIpcOpenMemHandle(&ptrs[i], b.h[i], cudaIpcMemLazyEnablePeerAccess);
                if (e != cudaSuccess) {
                    set_error("dsp_comm_connect: cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(e));
                    cudaGetLastError();
                    return DSP_ERR_CUDA;
                }
                c->opened[i][r] = true;
            }
        }
        c->peer_win[0][r] = ptrs[0]; c->peer_win[1][r] = ptrs[1]; c->peer_ctrl[r] = (Ctrl*)ptrs[2];
    }
    c->connected = true;
    return DSP_OK;
}

int dsp_comm_destroy(dsp_comm c) {
    if (!c) return DSP_OK;
    DevGuard g(c->device);
    cudaDeviceSynchronize();
    for (int r = 0; r < c->world; ++r) {
        if (c->opened[0][r]) cudaIpcCloseMemHandle(c->peer_win[0][r]);
        if (c->opened[1][r]) cudaIpcCloseMemHandle(c->peer_win[1][r]);
        if (c->opened[2][r]) cudaIpcCloseMemHandle(c->peer_ctrl[r]);
    }
    for (int w = 0; w < 2; ++w) if (c->win[w]) cudaFree(c->win[w]);
    if (c->ctrl) cudaFree(c->ctrl);
    if (c->d_tg) cudaFree(c->d_tg);
    if (c->d_abort) cudaFree(c->d_abort);
    if (c->d_res) cudaFree(c->d_res);
    if (c->h_res) cudaFreeHost(c->h_res);
    if (c->d_bounds) cudaFree(c->d_bounds);
    if (c->h_bounds) cudaFreeHost(c->h_bounds);
    for (int i = 0; i < 5; ++i) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    for (int i = 0; i < 10; ++i) if (c->dev[i / 5][i % 5]) cudaEventDestroy(c->dev[i / 5][i % 5]);
    cudaGetLastError();
    delete c;
    return DSP_OK;
}

int dsp_comm_route_rows(dsp_comm c, const void* rows, int64_t n, int32_t row_bytes, int32_t field_offset,
                        const uint64_t* bounds_host, void* out, int64_t out_cap_rows, int64_t* n_out_host, void* stream) {
    DSP_REQUIRE(c && n_out_host && bounds_host, DSP_ERR_INVALID, "dsp_comm_route_rows: null argument");
    *n_out_host = 0;
    DSP_REQUIRE(n >= 0 && (n == 0 || rows), DSP_ERR_INVALID, "dsp_comm_route_rows: bad rows");
    DSP_REQUIRE((row_bytes == 48 || row_bytes == 96) && field_offset >= 0 && field_offset % 8 == 0 && field_offset + 8 <= row_bytes,
                DSP_ERR_INVALID, "dsp_comm_route_rows: rows of 48 or 96 bytes, 8-byte aligned field");
    DevGuard g(c->device);
    cudaStream_t st = (cudaStream_t)stream;
    Scratch sc(c->device);
    int64_t got = 0;
    int rc = row_bytes == 48 ? route_rows_units<3>(c, sc, st, rows, n, field_offset / 8, bounds_host, &got)
                             : route_rows_units<6>(c, sc, st, rows, n, field_offset / 8, bounds_host, &got);
    if (rc) return rc;
    *n_out_host = got;
    DSP_REQUIRE(got <= out_cap_rows, DSP_ERR_NOMEM, "dsp_comm_route_rows: %lld rows received, capacity %lld", (long long)got, (long long)out_cap_rows);
    if (got) DSP_CUDA(cudaMemcpyAsync(out, c->win[1], (size_t)got * row_bytes, cudaMemcpyDeviceToDevice, st));
    DSP_CUDA(cudaStreamSynchronize(st));
    return DSP_OK;
}

int dsp_freq_aggregate_distributed(dsp_comm c, const uint64_t* key, const double* p0, const double* p1, const int32_t* label,
                                   int64_t n, uint64_t gidx_base, double prob_cf, const uint64_t* gidx_bounds_host,
                                   int32_t row_placement, void* rows_out, int64_t rows_cap, int64_t* n_rows_host,
                                   int64_t* n_callable_host, uint64_t* row_bounds_host, void* stream) {
    DSP_REQUIRE(c && n_rows_host && gidx_bounds_host, DSP_ERR_INVALID, "dsp_freq_aggregate_distributed: null argument");
    *n_rows_host = 0;
    if (n_callable_host) *n_callable_host = 0;
    DSP_REQUIRE(n >= 0 && n < (int64_t)0x7fffffff, DSP_ERR_INVALID, "dsp_freq_aggregate_distributed: n=%lld out of range", (long long)n);
    DSP_REQUIRE(n == 0 || (key && p0 && p1 && label), DSP_ERR_INVALID, "dsp_freq_aggregate_distributed: null column");
    DevGuard g(c->device);
    cudaStream_t st = (cudaStream_t)stream;
    Scratch sc(c->device);
    int rc;
    DSP_CUDA(cudaEventRecord(c->ev[0], st));
    // 1. callable records -> hash(key) % world, straight into the owners' windows
    route::RecFromColumns src{key, p0, p1, label, gidx_base, prob_cf, c->world};
    int64_t m = 0;
    unsigned long long bits = 0;
    if ((rc = exchange<route::RecFromColumns>(c, sc, st, src, n, 0, sizeof(Rec), &m, &bits))) return rc;
    if (n_callable_host) *n_callable_host = m;
    DSP_CUDA(cudaEventRecord(c->ev[1], st));
    // 2. my keys: sort + ordered replay (rows in key order)
    SiteRow* rows = nullptr;
    int64_t nseg = 0;
    if ((rc = sc.alloc(&rows, m))) return rc;
    if ((rc = sites_from_records(sc, st, reinterpret_cast<const Rec*>(c->win[0]), m, bits, rows, &nseg))) return rc;
    DSP_CUDA(cudaEventRecord(c->ev[2], st));
    // 3. rows -> the rank that owns the range of `first` (global index of the site's first callable record) they fall
    //    into: ranges of equal row count chosen from samples (row_placement 0), or the ranks' own record shards
    //    (row_placement 1: a row ends up where its first callable record was parsed)
    int64_t home = 0;
    if (row_placement == 0 && (rc = choose_row_splitters(c, st, rows, nseg))) return rc;
    if ((rc = route_rows_units<3>(c, sc, st, rows, nseg, 1, row_placement == 0 ? nullptr : gidx_bounds_host, &home))) return rc;
    if (row_bounds_host) {
        DSP_CUDA(cudaMemcpyAsync(c->h_bounds, c->d_bounds, sizeof(uint64_t) * (c->world + 1), cudaMemcpyDeviceToHost, st));
        DSP_CUDA(cudaStreamSynchronize(st));
        for (int w = 0; w <= c->world; ++w) row_bounds_host[w] = c->h_bounds[w];
    }
    DSP_CUDA(cudaEventRecord(c->ev[3], st));
    *n_rows_host = home;
    DSP_REQUIRE(home <= rows_cap, DSP_ERR_NOMEM, "dsp_freq_aggregate_distributed: %lld site rows, capacity %lld", (long long)home, (long long)rows_cap);
    // 4. dict insertion order on this rank = ascending first record
    int end_bit = 1;                                  // `first` is a global record index < bounds[world]
    while (end_bit < 63 && (1ull << end_bit) < gidx_bounds_host[c->world]) ++end_bit;
    if ((rc = sort_rows(sc, st, reinterpret_cast<const SiteRow*>(c->win[1]), home, 0, reinterpret_cast<SiteRow*>(rows_out), end_bit))) return rc;
    DSP_CUDA(cudaEventRecord(c->ev[4], st));
    DSP_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < 4; ++i) cudaEventElapsedTime(&c->last_ms[i], c->ev[i], c->ev[i + 1]);
    return DSP_OK;
}

int dsp_comm_allreduce_f32(dsp_comm c, float* const* bufs, const int64_t* numel, int32_t n_bufs, void* stream) {
    DSP_REQUIRE(n_bufs >= 0, DSP_ERR_INVALID, "dsp_comm_allreduce_f32: n_bufs=%d", (int)n_bufs);
    DSP_REQUIRE(n_bufs == 0 || (bufs && numel), DSP_ERR_INVALID, "dsp_comm_allreduce_f32: null buffer or size list");
    int64_t e = 0;
    for (int32_t i = 0; i < n_bufs; ++i) {
        DSP_REQUIRE(numel[i] >= 0 && numel[i] <= ((int64_t)1 << 40) - e, DSP_ERR_INVALID,
                    "dsp_comm_allreduce_f32: numel[%d]=%lld out of range", (int)i, (long long)numel[i]);
        DSP_REQUIRE(numel[i] == 0 || bufs[i], DSP_ERR_INVALID, "dsp_comm_allreduce_f32: bufs[%d] is null", (int)i);
        e += numel[i];
    }
    DSP_REQUIRE(c, DSP_ERR_INVALID, "dsp_comm_allreduce_f32: null communicator");
    DSP_REQUIRE(c->connected, DSP_ERR_STATE, "dsp_comm_allreduce_f32: not connected (dsp_comm_connect after exchanging the export blobs)");
    const int world = c->world, me = c->rank;
    const int64_t chunk = ar_chunk(e, world);
    DSP_REQUIRE(chunk * world * 4 <= c->window_bytes, DSP_ERR_NOMEM,
                "dsp_comm_allreduce_f32: %lld floats need windows of %lld bytes, the communicator has %lld",
                (long long)e, (long long)(chunk * world * 4), (long long)c->window_bytes);
    if (e == 0 || world == 1) return DSP_OK;
    DevGuard g(c->device);
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned long long epoch = ++c->epoch;
    Peers peers{}; Windows w0{}, w1{};
    for (int r = 0; r < world; ++r) { peers.ctrl[r] = c->peer_ctrl[r]; w0.win[r] = c->peer_win[0][r]; w1.win[r] = c->peer_win[1][r]; }
    auto blocks = [&](int64_t items, int per_sm) { return (int)std::max<int64_t>(1, std::min<int64_t>((items + AR_THREADS - 1) / AR_THREADS, (int64_t)c->n_sm * per_sm)); };
    DSP_CUDA(cudaMemsetAsync(c->d_abort, 0, sizeof(int), st));
    DSP_CUDA(cudaMemsetAsync(c->d_res, 0, sizeof(Result), st));
    std::vector<ArList> groups;
    int64_t o = 0;
    for (int32_t i0 = 0; i0 < n_bufs; i0 += AR_MAXT) {
        ArList l{};
        l.count = std::min<int32_t>(AR_MAXT, n_bufs - i0);
        for (int k = 0; k < l.count; ++k) { l.ptr[k] = bufs[i0 + k]; l.off[k] = o; o += numel[i0 + k]; }
        l.off[l.count] = o;
        groups.push_back(l);
    }
    for (const ArList& l : groups)
        if (l.off[l.count] > l.off[0]) allreduce_pack_kernel<<<blocks(l.off[l.count] - l.off[0], 8), AR_THREADS, 0, st>>>(l, w0, me, chunk);
    allreduce_signal_wait_kernel<<<1, 32, 0, st>>>(c->ctrl, peers, me, world, 0, epoch, c->d_abort, c->d_res);
    const int64_t lo = std::min<int64_t>(e, me * chunk), len = std::min<int64_t>(e, lo + chunk) - lo;
    if (len > 0)
        allreduce_reduce_kernel<<<blocks(len / 4 + 1, 4), AR_THREADS, 0, st>>>(static_cast<const float*>(c->win[0]), w1, world, chunk,
                                                                                 lo, len, c->d_abort);
    allreduce_signal_wait_kernel<<<1, 32, 0, st>>>(c->ctrl, peers, me, world, 1, epoch, c->d_abort, c->d_res);
    for (const ArList& l : groups)
        if (l.off[l.count] > l.off[0])
            allreduce_unpack_kernel<<<blocks(l.off[l.count] - l.off[0], 8), AR_THREADS, 0, st>>>(l, static_cast<const float*>(c->win[1]),
                                                                                               c->d_abort);
    DSP_CUDA(cudaGetLastError());
    DSP_CUDA(cudaMemcpyAsync(c->h_res, c->d_res, sizeof(Result), cudaMemcpyDeviceToHost, st));
    DSP_CUDA(cudaStreamSynchronize(st));
    DSP_REQUIRE(!(c->h_res->err & 2), DSP_ERR_CUDA, "dsp_comm_allreduce_f32: rank %d timed out waiting for a peer (call %llu)", me, epoch);
    return DSP_OK;
}

int dsp_comm_last_timing(dsp_comm c, float* ms12) {
    DSP_REQUIRE(c && ms12, DSP_ERR_INVALID, "dsp_comm_last_timing: null argument");
    for (int i = 0; i < 4; ++i) ms12[i] = c->last_ms[i];
    for (int i = 0; i < 8; ++i) ms12[4 + i] = c->detail_ms[i / 4][i % 4];
    return DSP_OK;
}

}  // extern "C"
