// Reconstruction F1 over all ordered node pairs without materialising the energies (check_graph_embedding,
// order_embeddings.py:512-559 = oe.py:1923-1990: the energy of every closure edge against that of every other ordered
// pair u != v, then EmbeddingMetrics.calculate_metrics('val')).
//
// The energies are the SIMT scoring kernel's (score_fast_kernel's Pass::F1: same per-pair instructions, so the same bits
// as the lec_score_topk_ex matrix), classified by the Euler intervals and counted, never stored (Pass::F1Dag: a DAG's
// interval cover, the Euler-like primary interval plus each apex's extra intervals; Pass::F1Held, F1HeldDag: positives
// only where the closure slot is held out, other closure pairs skipped):
//   round 0      every pair's key (fp32 bits; energies are >= 0 or NaN) into 2 x 32 768 coarse bins (key >> 16)
//   select       exact F1 at each coarse bin's largest value gives a lower bound LB on the best F1; a bin can
//                only hold a better threshold if 2 CP_b / (n_pos + CP_b + FP_{b-1}) >= LB (1 - 1e-12) -- the slack
//                covers the fp64 rounding of the reference's 2pr / (p + r) -- and only those bins are opened
//   round k      the energies again; pairs in the open bins are counted per exact key (65 536 fine bins each)
//   finish       every distinct value of the open bins is a threshold with exact cp / cn: lec_f1.cuh's f1_row,
//                first arg-max, carried across rounds when more bins are open than the workspace holds
// At a fixed threshold t (lec_recon_finish_at) round 0 gives the counts below key(t)'s coarse bin and one fine round,
// with only that bin open, the counts inside it up to key(t).
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

// exclusive prefix sum over the block (NT threads, NT / 32 <= 32 warps).  Not cub::BlockScan: cub's headers add device
// globals to this file, which would move the constant-bank slots the evaluation passes read their math tables from.
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

// the block's best candidate (f1_better: the higher F1, the lower key on a tie), in every thread
__device__ ReconBest block_best(ReconBest b) {
    __shared__ ReconBest sh[kSelThreads];
    const int tid = threadIdx.x;
    sh[tid] = b;
    __syncthreads();
    for (int w = kSelThreads / 2; w > 0; w >>= 1) {
        if (tid < w) {
            const ReconBest c = sh[tid + w], a = sh[tid];
            if (c.has && (!a.has || f1_better(c.f1, c.key, a.f1, a.key))) sh[tid] = c;
        }
        __syncthreads();
    }
    return sh[0];
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
    b = block_best(b);
    if (tid == 0) best[blockIdx.x] = b;
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
    const ReconBest c = block_best(b);
    if (tid == 0) {
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

// fixed threshold t (lec_recon_finish_at) after round 0: the finite pairs in the coarse bins below key(t)'s; that bin is
// opened for one fine round unless it is empty or t decides every pair by itself (NaN, below 0); one block
__global__ void __launch_bounds__(kSelThreads) recon_at_select_kernel(const u64c* __restrict__ hdr, const u64c* __restrict__ hist,
                                                                      ReconState* __restrict__ s, ReconOpen* __restrict__ open,
                                                                      int64_t batch, float t, double* __restrict__ out7,
                                                                      long long* __restrict__ status) {
    constexpr int PER = kReconBins / kSelThreads;
    if (s->phase != 0) return;
    const int tid = threadIdx.x;
    const u64c n_pos = hdr[0], n_neg = hdr[1], nan_neg = hdr[3];
    const unsigned bits = __float_as_uint(t);
    const bool nan_t = t != t, neg_t = !nan_t && bits > 0x80000000u;  // -0 is 0
    const int bin = nan_t || neg_t ? 0 : (int)((bits & 0x7fffffffu) >> kReconShift);
    const u64c* hp = hist;
    const u64c* hn = hist + kReconBins;
    u64c sp = 0, sn = 0;
    for (int j = 0; j < PER; ++j) {
        const int b = tid * PER + j;
        if (b < bin) { sp += hp[b]; sn += hn[b]; }
    }
    u64c cp, fp;
    block_exclusive_scan<u64c, kSelThreads>(sp, cp);
    block_exclusive_scan<u64c, kSelThreads>(sn, fp);   // finite negatives below the bin
    if (tid == 0) {
        const bool fine = !nan_t && !neg_t && (hp[bin] | hn[bin]) != 0;
        s->n_pos = n_pos; s->n_neg = n_neg; s->nan_pos = hdr[2]; s->nan_neg = nan_neg;
        s->batch = batch; s->n_open = fine; s->next = 0; s->m = fine;
        s->phase = fine ? 1 : 2;
        s->has_best = 0;
        status[0] = fine; status[1] = fine; status[2] = (long long)n_pos; status[3] = (long long)n_neg;
        if (fine) open[0] = ReconOpen{(uint32_t)bin, 0u, cp, fp};
        else if (nan_t) f1_row_at(t, 0, 0, (int64_t)n_pos, (int64_t)n_neg, out7);   // no comparison with NaN holds
        else f1_row_at(t, (int64_t)cp, (int64_t)(n_neg - nan_neg - fp), (int64_t)n_pos, (int64_t)n_neg, out7);
    }
}

// fixed threshold, fine round: the exact values of key(t)'s coarse bin up to key(t); one block
__global__ void __launch_bounds__(kSelThreads) recon_at_fine_kernel(const u64c* __restrict__ hist, ReconState* __restrict__ s,
                                                                    const ReconOpen* __restrict__ open, float t,
                                                                    double* __restrict__ out7, long long* __restrict__ status) {
    constexpr int PER = kReconFine / kSelThreads;
    const int tid = threadIdx.x;
    const int phase = s->phase;
    if (phase != 1) {
        if (phase == 2 && tid == 0) { status[0] = 0; status[1] = s->n_open; status[2] = (long long)s->n_pos; status[3] = (long long)s->n_neg; }
        return;
    }
    const int low = (int)(__float_as_uint(t) & 0x7fffffffu & (kReconFine - 1));   // t is >= 0 here; -0 is 0
    const u64c* h = hist;   // batch slot 0: [fine][negative, positive]
    u64c sp = 0, sn = 0;
    for (int j = 0; j < PER; ++j) {
        const int f = tid * PER + j;
        if (f <= low) { sp += h[2 * f + 1]; sn += h[2 * f]; }
    }
    u64c cp, fp;
    block_exclusive_scan<u64c, kSelThreads>(sp, cp);
    block_exclusive_scan<u64c, kSelThreads>(sn, fp);
    if (tid == 0) {
        const ReconOpen o = open[0];
        const ReconState st = *s;
        cp += o.cp_below;
        fp += o.fp_below;
        f1_row_at(t, (int64_t)cp, (int64_t)(st.n_neg - st.nan_neg - fp), (int64_t)st.n_pos, (int64_t)st.n_neg, out7);
        s->next = 1; s->m = 0; s->phase = 2;
        status[0] = 0; status[1] = 1; status[2] = (long long)st.n_pos; status[3] = (long long)st.n_neg;
    }
}

int validate(const lec_recon_t* r) {
    return eval_validate(r, true, [&] { return batch_of(r->workspace_bytes) < 1 ? LEC_E_SIZE : 0; });
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

extern "C" int lec_recon_pass_heldout(const lec_recon_t* r, const lec_recon_extra_t* x, const lec_heldout_t* h,
                                      void* stream) {
    using namespace lec;
    const int err = validate(r);
    if (err) return err;
    const bool dag = x != nullptr && x->count != 0;
    if (dag) {
        if (x->count < 0 || x->count > 0x7fffffffLL) return LEC_E_SIZE;
        if (!x->ptr || !x->lo || !x->hi) return LEC_E_NULL;
    }
    if (h) {
        const int herr = heldout_validate(h, dag);
        if (herr) return herr;
        if (dag && x->count > h->n_closure) return LEC_E_SIZE;   // an extra interval holds at least one closure pair
    }
    if (r->u_end == r->u_begin) return 0;
    const Layout l = layout(r->workspace, r->workspace_bytes);
    FastArgs a{};
    a.labels = r->rows; a.images = r->rows; a.L = r->n; a.N = r->n; a.D = r->D; a.K = r->K; a.k = 1;
    a.ld = r->ld; a.u_begin = r->u_begin; a.u_end = r->u_end;
    a.tin = r->tin; a.tout = r->tout;
    a.rstate = l.state; a.ropen = l.open; a.rhdr = l.hdr; a.rhist = l.hist;
    if (dag) { a.xptr = x->ptr; a.xlo = x->lo; a.xhi = x->hi; }
    if (h) { a.hptr = h->closure_ptr; a.hmap = h->slot_map; a.rxcum = h->xcum; }
    cudaStream_t st = (cudaStream_t)stream;
    // only apexes with extra intervals leave the forest pass's instructions; only pairs below their apex look up the
    // slot map
    if (h) return dag ? eval_launch<Pass::F1HeldDag>(r->geom, a, st) : eval_launch<Pass::F1Held>(r->geom, a, st);
    return dag ? eval_launch<Pass::F1Dag>(r->geom, a, st) : eval_launch<Pass::F1>(r->geom, a, st);
}

extern "C" int lec_recon_pass_dag(const lec_recon_t* r, const lec_recon_extra_t* x, void* stream) {
    return lec_recon_pass_heldout(r, x, nullptr, stream);
}

extern "C" int lec_recon_pass(const lec_recon_t* r, void* stream) {
    return lec_recon_pass_dag(r, nullptr, stream);
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

extern "C" int lec_recon_finish_at(const lec_recon_t* r, float threshold, double* out7, int64_t* status, void* stream) {
    using namespace lec;
    const int err = validate(r);
    if (err) return err;
    if (!out7 || !status) return LEC_E_NULL;
    const Layout l = layout(r->workspace, r->workspace_bytes);
    cudaStream_t st = (cudaStream_t)stream;
    // as lec_recon_finish: the fine-round kernel returns at once unless the fine round is being finished, the round-0
    // kernel unless round 0 is
    recon_at_fine_kernel<<<1, kSelThreads, 0, st>>>(l.hist, l.state, l.open, threshold, out7, reinterpret_cast<long long*>(status));
    recon_at_select_kernel<<<1, kSelThreads, 0, st>>>(l.hdr, l.hist, l.state, l.open, l.batch, threshold, out7,
                                                       reinterpret_cast<long long*>(status));
    g_launches += 2;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    return (int)cudaMemsetAsync(r->workspace, 0, (size_t)l.counter_bytes, st);
}
