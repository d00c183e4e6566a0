// Reconstruction F1 over all ordered node pairs without materialising the energies (check_graph_embedding,
// order_embeddings.py:512-559 = oe.py:1923-1990: the energy of every closure edge against that of every other ordered
// pair u != v, then EmbeddingMetrics.calculate_metrics('val')).
//
// The energies are the SIMT scoring kernel's (score_fast_kernel with EPI = 1: same per-pair instructions, so the same
// bits as the lec_score_topk_ex matrix), classified by the Euler intervals and counted, never stored:
//   round 0      every pair's key (fp32 bits; energies are >= 0 or NaN) into 2 x 32 768 coarse bins (key >> 16)
//   select       exact F1 at each coarse bin's largest value gives a lower bound LB on the best F1; a bin can
//                only hold a better threshold if 2 CP_b / (n_pos + CP_b + FP_{b-1}) >= LB (1 - 1e-12) -- the slack
//                covers the fp64 rounding of the reference's 2pr / (p + r) -- and only those bins are opened
//   round k      the energies again; pairs in the open bins are counted per exact key (65 536 fine bins each)
//   finish       every distinct value of the open bins is a threshold with exact cp / cn: lec_f1.cuh's f1_row,
//                first arg-max, carried across rounds when more bins are open than the workspace holds
//
// Workspace (caller-owned, zeroed once before round 0):
//   [counters]  8 x u64 header {n_pos, n_neg, NaN positives, NaN negatives} + batch x 2 x 65 536 u64 histogram
//               (round 0 uses its first 2 x 32 768 words); what ranks sum after a pass, cleared by every finish
//   [state]     ReconState (round, open-bin batch, best so far)
//   [open]      32 768 x ReconOpen: the open coarse bins in key order with the finite counts below each
//   [best]      batch x ReconBest: per-open-bin winners of a fine round
#include "lec_f1.cuh"
#include "lec_score_fast_impl.cuh"

namespace lec {
namespace {

typedef unsigned long long u64c;
// one block per SM (128 KB of shared counters): 16 warps where the image rows fit 128 registers, else 8 (D > 32 spills
// at 512 threads)
template <int DH>
constexpr int recon_threads() { return DH > 16 ? 256 : 512; }
constexpr int kReconTarget = 148 * 16;  // blocks per pass to aim for (16 waves: the chunks balance)
constexpr int64_t kReconMaxChunk = 4096;  // apex rows per block: its 32-bit shared counters cannot overflow
constexpr int kSelThreads = 1024;
constexpr int64_t kMaxBatch = 16383;  // fine tags (slot, key, sign) fit an int

struct ReconBest { double f1; u64c cp, cn; unsigned key; int has; };

constexpr int64_t kHdrBytes = 64;
constexpr int64_t kStateBytes = 256;
constexpr int64_t kOpenBytes = (int64_t)kReconBins * sizeof(ReconOpen);
constexpr int64_t kPerBinBytes = 2 * (int64_t)kReconFine * 8 + sizeof(ReconBest);
constexpr int64_t kFixedBytes = kHdrBytes + kStateBytes + kOpenBytes;
static_assert(sizeof(ReconState) <= kStateBytes, "state");
static_assert(2 * kReconBins <= 2 * kReconFine, "a fine slot holds the coarse histogram");

int64_t batch_of(int64_t ws_bytes) {
    if (ws_bytes < kFixedBytes + kPerBinBytes) return 0;
    const int64_t b = (ws_bytes - kFixedBytes) / kPerBinBytes;
    return b < kMaxBatch ? b : kMaxBatch;
}
int64_t counter_bytes_of(int64_t batch) { return kHdrBytes + batch * 2 * (int64_t)kReconFine * 8; }

struct Layout {
    u64c* hdr; u64c* hist; ReconState* state; ReconOpen* open; ReconBest* best; int64_t batch, counter_bytes;
};
Layout layout(void* ws, int64_t ws_bytes) {
    Layout l;
    l.batch = batch_of(ws_bytes);
    l.counter_bytes = counter_bytes_of(l.batch);
    char* p = static_cast<char*>(ws);
    l.hdr = reinterpret_cast<u64c*>(p);
    l.hist = reinterpret_cast<u64c*>(p + kHdrBytes);
    l.state = reinterpret_cast<ReconState*>(p + l.counter_bytes);
    l.open = reinterpret_cast<ReconOpen*>(p + l.counter_bytes + kStateBytes);
    l.best = reinterpret_cast<ReconBest*>(p + l.counter_bytes + kStateBytes + kOpenBytes);
    return l;
}

// exclusive prefix sum over the block (NT threads, NT / 32 <= 32 warps)
template <typename T, int NT>
__device__ T block_exclusive_scan(T x, T& total) {
    __shared__ T warp_sum[NT / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    T inc = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    __syncthreads();
    if (lane == 31) warp_sum[w] = inc;
    __syncthreads();
    if (w == 0) {
        T s = lane < NT / 32 ? warp_sum[lane] : T(0);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        if (lane < NT / 32) warp_sum[lane] = s;  // inclusive over warps
    }
    __syncthreads();
    total = warp_sum[NT / 32 - 1];
    const T before = w > 0 ? warp_sum[w - 1] : T(0);
    return before + inc - x;
}

__device__ void write_row(const ReconState& s, float t, u64c cp, u64c cn, double* out7) {
    f1_row(t, (int64_t)cp, (int64_t)cn, (int64_t)s.n_pos, (int64_t)s.n_neg, out7);
}

// after round 0: totals, lower bound, open list; one block
__global__ void __launch_bounds__(kSelThreads) recon_select_kernel(const u64c* __restrict__ hdr, const u64c* __restrict__ hist,
                                                                   ReconState* __restrict__ s, ReconOpen* __restrict__ open,
                                                                   int64_t batch, double* __restrict__ out7, long long* __restrict__ status) {
    constexpr int PER = kReconBins / kSelThreads;
    if (s->phase != 0) return;
    const int tid = threadIdx.x;
    const u64c n_pos = hdr[0], n_neg = hdr[1], nan_neg = hdr[3];
    const u64c* hp = hist;
    const u64c* hn = hist + kReconBins;
    u64c sp = 0, sn = 0;
    for (int j = 0; j < PER; ++j) { sp += hp[tid * PER + j]; sn += hn[tid * PER + j]; }
    u64c tot;
    const u64c cp0 = block_exclusive_scan<u64c, kSelThreads>(sp, tot);
    const u64c fp0 = block_exclusive_scan<u64c, kSelThreads>(sn, tot) + nan_neg;  // fp counts NaN negatives (E > t fails)
    // LB = best exact F1 at a bin's largest value = 2 CP_b / (n_pos + CP_b + FP_b); first non-empty bin
    double lb = 0.0;
    int first = kReconBins;
    u64c cp = cp0, fp = fp0;
    for (int j = 0; j < PER; ++j) {
        const int b = tid * PER + j;
        const u64c p = hp[b], q = hn[b];
        if ((p | q) == 0) continue;
        cp += p; fp += q;
        first = min(first, b);
        lb = fmax(lb, 2.0 * (double)cp / (double)(n_pos + cp + fp));
    }
    __shared__ double s_lb[kSelThreads / 32];
    __shared__ int s_first[kSelThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lb = fmax(lb, __shfl_xor_sync(0xffffffffu, lb, o));
        first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
    }
    if ((tid & 31) == 0) { s_lb[tid >> 5] = lb; s_first[tid >> 5] = first; }
    __syncthreads();
    for (int w = 0; w < kSelThreads / 32; ++w) { lb = fmax(lb, s_lb[w]); first = min(first, s_first[w]); }
    // open: every bin whose upper bound reaches LB; with LB = 0 (no positive can be classified) every threshold
    // scores 0 or NaN and the lowest one wins, so only the first bin is opened
    const double cut = lb * (1.0 - 1e-12);
    unsigned flags = 0;
    int cnt = 0;
    cp = cp0; fp = fp0;
    for (int j = 0; j < PER; ++j) {
        const int b = tid * PER + j;
        const u64c p = hp[b], q = hn[b];
        if ((p | q) == 0) continue;
        const double ub = 2.0 * (double)(cp + p) / (double)(n_pos + cp + p + fp);
        if (lb > 0.0 ? ub >= cut : b == first) { flags |= 1u << j; ++cnt; }
        cp += p; fp += q;
    }
    int n_open;
    int at = block_exclusive_scan<int, kSelThreads>(cnt, n_open);
    cp = cp0; fp = fp0 - nan_neg;
    for (int j = 0; j < PER; ++j) {
        const int b = tid * PER + j;
        if (flags & (1u << j)) open[at++] = ReconOpen{(uint32_t)b, 0u, cp, fp};
        cp += hp[b]; fp += hn[b];
    }
    if (tid == 0) {
        s->n_pos = n_pos; s->n_neg = n_neg; s->nan_pos = hdr[2]; s->nan_neg = nan_neg;
        s->batch = batch; s->n_open = n_open; s->next = 0; s->m = n_open < batch ? n_open : batch;
        s->phase = n_open > 0 ? 1 : 2;
        s->has_best = 0;
        status[0] = n_open > 0; status[1] = n_open; status[2] = (long long)n_pos; status[3] = (long long)n_neg;
        if (n_open == 0) {  // no finite energy: the NaN threshold is the only candidate (or there is no pair at all)
            if (n_pos + n_neg == 0) { for (int j = 0; j < 7; ++j) out7[j] = nan(""); }
            else write_row(*s, __int_as_float(0x7fc00000), 0, 0, out7);
        }
    }
}

// fine round: block i walks the 65 536 exact values of open bin next + i in key order
__global__ void __launch_bounds__(kSelThreads) recon_fine_kernel(const u64c* __restrict__ hist, const ReconState* __restrict__ s,
                                                                 const ReconOpen* __restrict__ open, ReconBest* __restrict__ best) {
    constexpr int PER = kReconFine / kSelThreads;
    if (s->phase != 1 || blockIdx.x >= s->m) return;
    const int tid = threadIdx.x;
    const ReconOpen o = open[s->next + blockIdx.x];
    const u64c* h = hist + (size_t)blockIdx.x * kReconFine * 2;   // [fine][negative, positive]
    const ReconState st = *s;
    u64c sp = 0, sn = 0;
    for (int j = 0; j < PER; ++j) { sp += h[2 * (tid * PER + j) + 1]; sn += h[2 * (tid * PER + j)]; }
    u64c tot;
    u64c cp = o.cp_below + block_exclusive_scan<u64c, kSelThreads>(sp, tot);
    u64c fp = o.fp_below + block_exclusive_scan<u64c, kSelThreads>(sn, tot);   // finite negatives <= t
    const u64c neg_fin = st.n_neg - st.nan_neg;
    ReconBest b{-1.0, 0, 0, 0u, 0};
    for (int j = 0; j < PER; ++j) {
        const int f = tid * PER + j;
        const u64c p = h[2 * f + 1], q = h[2 * f];
        if ((p | q) == 0) continue;
        cp += p; fp += q;
        const unsigned key = (o.bin << kReconShift) | (unsigned)f;
        double row[7];
        write_row(st, __uint_as_float(key), cp, neg_fin - fp, row);
        const double f1 = row[0] == row[0] ? row[0] : -1.0;   // NaN never wins
        if (!b.has || f1 > b.f1) b = ReconBest{f1, cp, neg_fin - fp, key, 1};
    }
    __shared__ ReconBest sh[kSelThreads];
    sh[tid] = b;
    __syncthreads();
    for (int w = kSelThreads / 2; w > 0; w >>= 1) {
        if (tid < w) {
            const ReconBest c = sh[tid + w], a = sh[tid];
            if (c.has && (!a.has || f1_better(c.f1, c.key, a.f1, a.key))) sh[tid] = c;
        }
        __syncthreads();
    }
    if (tid == 0) best[blockIdx.x] = sh[0];
}

// end of a fine round: merge the batch into the carried best (earlier batches hold lower keys: they win ties)
__global__ void __launch_bounds__(kSelThreads) recon_merge_kernel(ReconState* __restrict__ s, const ReconBest* __restrict__ best,
                                                                  double* __restrict__ out7, long long* __restrict__ status) {
    const int tid = threadIdx.x;
    if (s->phase != 1) {
        if (s->phase == 2 && tid == 0) { status[0] = 0; status[1] = s->n_open; status[2] = (long long)s->n_pos; status[3] = (long long)s->n_neg; }
        return;
    }
    const long long m = s->m;
    ReconBest b{-1.0, 0, 0, 0u, 0};
    for (long long i = tid; i < m; i += kSelThreads) {
        const ReconBest c = best[i];
        if (c.has && (!b.has || f1_better(c.f1, c.key, b.f1, b.key))) b = c;
    }
    __shared__ ReconBest sh[kSelThreads];
    sh[tid] = b;
    __syncthreads();
    for (int w = kSelThreads / 2; w > 0; w >>= 1) {
        if (tid < w) {
            const ReconBest c = sh[tid + w], a = sh[tid];
            if (c.has && (!a.has || f1_better(c.f1, c.key, a.f1, a.key))) sh[tid] = c;
        }
        __syncthreads();
    }
    if (tid == 0) {
        const ReconBest c = sh[0];
        if (c.has && (!s->has_best || c.f1 > s->best_f1)) {
            s->best_f1 = c.f1; s->best_cp = c.cp; s->best_cn = c.cn; s->best_key = c.key; s->has_best = 1;
        }
        s->next += m;
        const long long left = s->n_open - s->next;
        s->m = left < s->batch ? left : s->batch;
        s->phase = left > 0 ? 1 : 2;
        status[0] = left > 0; status[1] = s->n_open; status[2] = (long long)s->n_pos; status[3] = (long long)s->n_neg;
        if (s->has_best) write_row(*s, __uint_as_float(s->best_key), s->best_cp, s->best_cn, out7);
    }
}

template <int GEOM, int DH, int RI>
int recon_launch_dh(FastArgs& a, cudaStream_t st) {
    constexpr int NT = recon_threads<DH>();
    constexpr int LS = 4 * ((DH + 1) / 2) + 8;
    const size_t smem = (size_t)kTileLabels * LS * sizeof(float) + (size_t)kReconBins * sizeof(unsigned);
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(score_fast_kernel<GEOM, DH, RI, NT, 1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        configured = true;
    }
    a.groups = (a.N + (int64_t)NT * RI - 1) / ((int64_t)NT * RI);
    const int64_t rows = a.u_end - a.u_begin;
    int64_t chunks = (kReconTarget + a.groups - 1) / a.groups;
    int64_t chunk = (rows + chunks - 1) / chunks;
    if (chunk < 32) chunk = 32;
    if (chunk > kReconMaxChunk) chunk = kReconMaxChunk;
    a.chunk = chunk;
    chunks = (rows + chunk - 1) / chunk;
    const int64_t blocks = a.groups * chunks;
    if (blocks > 0x7fffffffLL) return LEC_E_SIZE;
    score_fast_kernel<GEOM, DH, RI, NT, 1, 1><<<(unsigned)blocks, NT, smem, st>>>(a);
    ++g_launches;
    return (int)cudaGetLastError();
}

template <int GEOM>
int recon_launch_geom(FastArgs& a, cudaStream_t st) {
    const int dh = (a.D + 1) / 2;   // the scoring kernel's instantiations (fast_launch_geom)
    if (dh <= 1) return recon_launch_dh<GEOM, 1, 4>(a, st);
    if (dh <= 2) return recon_launch_dh<GEOM, 2, 4>(a, st);
    if (dh <= 5) return recon_launch_dh<GEOM, 5, 4>(a, st);
    if (dh <= 8) return recon_launch_dh<GEOM, 8, 4>(a, st);
    if (dh <= 16) return recon_launch_dh<GEOM, 16, 2>(a, st);
    if (dh <= 25) return recon_launch_dh<GEOM, 25, 2>(a, st);
    if (dh <= 32) return recon_launch_dh<GEOM, 32, 2>(a, st);
    return LEC_E_DIM;
}

int validate(const lec_recon_t* r) {
    if (!r || !r->rows || !r->tin || !r->tout || !r->workspace) return LEC_E_NULL;
    if (r->D < 1 || r->D > 64 || r->ld < r->D || (r->ld != r->D && r->ld % 4 != 0)) return LEC_E_DIM;
    if (r->geom != LEC_GEOM_EUC && r->geom != LEC_GEOM_HYP && r->geom != LEC_GEOM_OE) return LEC_E_ENUM;
    if (r->n < 0 || r->n > 0x7fffffffLL || r->u_begin < 0 || r->u_end < r->u_begin || r->u_end > r->n) return LEC_E_SIZE;
    if (batch_of(r->workspace_bytes) < 1) return LEC_E_SIZE;
    if ((reinterpret_cast<uintptr_t>(r->rows) & 15) || (reinterpret_cast<uintptr_t>(r->workspace) & 15)) return LEC_E_ALIGN;
    return 0;
}

}  // namespace
}  // namespace lec

extern "C" int64_t lec_recon_workspace_bytes(int open_bins_per_round) {
    using namespace lec;
    if (open_bins_per_round < 1 || open_bins_per_round > kMaxBatch) return LEC_E_SIZE;
    return kFixedBytes + (int64_t)open_bins_per_round * kPerBinBytes;
}

extern "C" int64_t lec_recon_counter_bytes(int64_t workspace_bytes) {
    const int64_t b = lec::batch_of(workspace_bytes);
    return b < 1 ? (int64_t)LEC_E_SIZE : lec::counter_bytes_of(b);
}

extern "C" int lec_recon_pass(const lec_recon_t* r, void* stream) {
    using namespace lec;
    const int err = validate(r);
    if (err) return err;
    if (r->u_end == r->u_begin) return 0;
    const Layout l = layout(r->workspace, r->workspace_bytes);
    FastArgs a{};
    a.labels = r->rows; a.images = r->rows; a.L = r->n; a.N = r->n; a.D = r->D; a.K = r->K; a.k = 1;
    a.ld = r->ld; a.u_begin = r->u_begin; a.u_end = r->u_end;
    a.tin = r->tin; a.tout = r->tout;
    a.rstate = l.state; a.ropen = l.open; a.rhdr = l.hdr; a.rhist = l.hist;
    cudaStream_t st = (cudaStream_t)stream;
    switch (r->geom) {
        case LEC_GEOM_EUC: return recon_launch_geom<LEC_GEOM_EUC>(a, st);
        case LEC_GEOM_HYP: return recon_launch_geom<LEC_GEOM_HYP>(a, st);
        default: return recon_launch_geom<LEC_GEOM_OE>(a, st);
    }
}

extern "C" int lec_recon_finish(const lec_recon_t* r, double* out7, int64_t* status, void* stream) {
    using namespace lec;
    const int err = validate(r);
    if (err) return err;
    if (!out7 || !status) return LEC_E_NULL;
    const Layout l = layout(r->workspace, r->workspace_bytes);
    cudaStream_t st = (cudaStream_t)stream;
    // The host does not know the round.  The fine-round kernels run first and return at once unless a fine round is
    // being finished; the select kernel then returns at once unless round 0 is; so the call never reads device state.
    recon_fine_kernel<<<(unsigned)l.batch, kSelThreads, 0, st>>>(l.hist, l.state, l.open, l.best);
    recon_merge_kernel<<<1, kSelThreads, 0, st>>>(l.state, l.best, out7, reinterpret_cast<long long*>(status));
    recon_select_kernel<<<1, kSelThreads, 0, st>>>(l.hdr, l.hist, l.state, l.open, l.batch, out7,
                                                    reinterpret_cast<long long*>(status));
    g_launches += 3;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    return (int)cudaMemsetAsync(r->workspace, 0, (size_t)l.counter_bytes, st);   // the next pass adds to zero
}
