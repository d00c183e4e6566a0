// Reconstruction mean rank and MAP over all ordered node pairs without materialising the energies (the ranking
// evaluation of Nickel & Kiela's Poincaré embeddings, over the pairs and energies of lec_recon.cu).  One call, four
// stages, no host round trip:
//   keys     score_fast_kernel<Pass::RankKeys>: the rank key of every positive pair into its slot pos_ptr[u] + slot(u, v)
//            (same <GEOM, DH, RI> as lec_recon_pass, so the same energy bits as the SIMT matrix)
//   sort     cub::DeviceSegmentedRadixSort of each apex's keys (31 key bits), carrying the slot ids.  Not
//            DeviceSegmentedSort: above 500 segments it copies its partition sizes to the host and synchronises.
//   count    score_fast_kernel<Pass::RankCounts>: a negative at or below its apex's largest positive key adds 1 to cnt[b] and,
//            when it equals sorted[b], to eq[b], where b is its lower bound among the apex's sorted keys
//   finish   per apex: rank_pess = 1 + prefix(cnt) at the slot, rank_opt = rank_pess - eq[first slot of its tie group],
//            AP_u in fp64 in a fixed order
// On a held-out set (lec_rank_run_heldout) pos_ptr is the held-out layout and the key pass is Pass::RankKeysHeld: it
// finds each positive's closure slot as RankKeys does and writes the key to the held-out slot the slot map gives, or nowhere.  Sort,
// count and finish run unchanged: the count already leaves out every closure pair, held out or not.
//
// Workspace (caller-owned, needs no initialisation; each region 256-byte aligned):
//   napex (int) | apex list int32[n] | xcum int32[n_pos] | keys, slot ids in and out (4 x 4 B x n_pos) |
//   cnt, eq uint32[n_pos] | the sort's temporary storage
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_segmented_radix_sort.cuh>

#include "lec_score_fast_impl.cuh"

namespace lec {
namespace {

constexpr int kRankPrepThreads = 1024;
constexpr int kRankFinishThreads = 256;
constexpr int kRankFinishBlocks = 148 * 8;
constexpr int kRankKeyBits = 31;  // keys are <= 0x7fc00000

size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

cudaError_t sort_temp_bytes(int64_t n, int64_t n_pos, size_t& bytes) {
    bytes = 0;
    return cub::DeviceSegmentedRadixSort::SortPairs(nullptr, bytes, (const unsigned*)nullptr, (unsigned*)nullptr,
                                                    (const int32_t*)nullptr, (int32_t*)nullptr, (int)n_pos, (int)n,
                                                    (const int64_t*)nullptr, (const int64_t*)nullptr, 0, kRankKeyBits);
}

struct RankLayout {
    int* napex; int32_t* apex; int32_t* xcum; unsigned* key_in; int32_t* val_in; unsigned* key_out; int32_t* val_out;
    unsigned* cnt; unsigned* eq; void* temp; size_t fixed;
};
RankLayout rank_layout(void* ws, int64_t n, int64_t n_pos) {
    RankLayout l;
    char* p = static_cast<char*>(ws);
    size_t o = 0;
    const size_t q = al256((size_t)n_pos * 4);
    l.napex = reinterpret_cast<int*>(p + o); o += 256;
    l.apex = reinterpret_cast<int32_t*>(p + o); o += al256((size_t)n * 4);
    l.xcum = reinterpret_cast<int32_t*>(p + o); o += q;
    l.key_in = reinterpret_cast<unsigned*>(p + o); o += q;
    l.val_in = reinterpret_cast<int32_t*>(p + o); o += q;
    l.key_out = reinterpret_cast<unsigned*>(p + o); o += q;
    l.val_out = reinterpret_cast<int32_t*>(p + o); o += q;
    l.cnt = reinterpret_cast<unsigned*>(p + o); o += q;
    l.eq = reinterpret_cast<unsigned*>(p + o); o += q;
    l.temp = p + o;
    l.fixed = o;
    return l;
}

// the apexes of [u_begin, u_end) with P_u >= 1, in order; one block
__global__ void __launch_bounds__(kRankPrepThreads) rank_apex_kernel(const int64_t* __restrict__ pos, int64_t u_begin,
                                                                     int64_t u_end, int32_t* __restrict__ apex,
                                                                     int* __restrict__ napex) {
    using Scan = cub::BlockScan<int, kRankPrepThreads>;
    __shared__ typename Scan::TempStorage tmp;
    int base = 0;
    for (int64_t u0 = u_begin; u0 < u_end; u0 += kRankPrepThreads) {
        const int64_t u = u0 + threadIdx.x;
        const int has = u < u_end && pos[u + 1] > pos[u];
        int off, tot;
        Scan(tmp).ExclusiveSum(has, off, tot);
        if (has) apex[base + off] = (int32_t)u;
        base += tot;
        __syncthreads();  // tmp is reused
    }
    if (threadIdx.x == 0) *napex = base;
}

// xcum[i] = slots before extra interval i of its apex: the primary interval's, then the earlier extra intervals'; a warp
// per apex
__global__ void rank_xcum_kernel(const int32_t* __restrict__ tin, const int32_t* __restrict__ tout,
                                 const int32_t* __restrict__ xptr, const int32_t* __restrict__ xlo,
                                 const int32_t* __restrict__ xhi, int64_t u_begin, int64_t u_end,
                                 int32_t* __restrict__ xcum) {
    const int64_t u = u_begin + ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
    const int lane = threadIdx.x & 31;
    if (u >= u_end) return;
    const int x0 = xptr[u], x1 = xptr[u + 1];
    int carry = tout[u] - tin[u];
    for (int i0 = x0; i0 < x1; i0 += 32) {
        const int i = i0 + lane;
        const int len = i < x1 ? xhi[i] - xlo[i] + 1 : 0;
        int inc = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        if (i < x1) xcum[i] = carry + inc - len;
        carry += __shfl_sync(0xffffffffu, inc, 31);
    }
}

// per apex of the list: ranks of its slots from the prefix of cnt, AP_u in a fixed order; blocks stride over the list
__global__ void __launch_bounds__(kRankFinishThreads) rank_finish_kernel(
    const int64_t* __restrict__ pos, const int32_t* __restrict__ apex, const int* __restrict__ napex,
    const unsigned* __restrict__ skey, const int32_t* __restrict__ sval, const unsigned* __restrict__ cnt,
    const unsigned* __restrict__ eq, unsigned long long* __restrict__ sums, double* __restrict__ ap,
    int32_t* __restrict__ ranks) {
    constexpr int NT = kRankFinishThreads;
    using ScanI = cub::BlockScan<int, NT>;
    using RedD = cub::BlockReduce<double, NT>;
    using RedL = cub::BlockReduce<long long, NT>;
    __shared__ union {
        typename ScanI::TempStorage scan;
        typename RedD::TempStorage red;
        typename RedL::TempStorage redl;
    } tmp;
    __shared__ int carry[2];
    const int tid = threadIdx.x;
    const int m = *napex;
    long long s_opt = 0, s_pess = 0, s_cnt = 0;
    for (int a = blockIdx.x; a < m; a += gridDim.x) {
        const int u = apex[a];
        const int64_t base = pos[u];
        const int P = (int)(pos[u + 1] - base);
        double ap_u = 0.0;
        int cc = 0, cf = 0;  // negatives counted before the chunk; first slot of the tie group open at its start
        for (int c0 = 0; c0 < P; c0 += NT) {
            const int j = c0 + tid;
            const bool ok = j < P;
            const unsigned k = ok ? skey[base + j] : 0u;
            const bool first = ok && (j == 0 || skey[base + j - 1] != k);
            const bool last = ok && (j == P - 1 || skey[base + j + 1] != k);
            int C, f;
            ScanI(tmp.scan).InclusiveSum(ok ? (int)cnt[base + j] : 0, C);
            __syncthreads();
            ScanI(tmp.scan).InclusiveScan(first ? j : -1, f, cub::Max());
            __syncthreads();
            C += cc;          // negatives with key <= key(j) (a tie group's later slots have empty buckets)
            f = max(f, cf);
            double term = 0.0;
            if (ok) {
                const int r_pess = 1 + C, r_opt = r_pess - (int)eq[base + f];
                s_opt += r_opt;
                s_pess += r_pess;
                if (ranks) {
                    const int64_t sl = sval[base + j];
                    ranks[2 * sl] = r_opt;
                    ranks[2 * sl + 1] = r_pess;
                }
                if (last) term = (double)(j - f + 1) * ((double)(j + 1) / (double)(j + 1 + C));
            }
            const double tsum = RedD(tmp.red).Sum(term);
            if (tid == NT - 1) { carry[0] = C; carry[1] = f; }
            if (tid == 0) ap_u += tsum;
            __syncthreads();
            cc = carry[0];
            cf = carry[1];
            __syncthreads();
        }
        if (tid == 0) {
            ap[u] = ap_u / (double)P;  // exactly 1 when no negative ranks above a positive
            s_cnt += cc;
        }
    }
    const long long t_opt = RedL(tmp.redl).Sum(s_opt);
    __syncthreads();
    const long long t_pess = RedL(tmp.redl).Sum(s_pess);
    __syncthreads();
    const long long t_cnt = RedL(tmp.redl).Sum(s_cnt);
    if (tid == 0) {
        if (t_opt) atomicAdd(sums + 0, (unsigned long long)t_opt);
        if (t_pess) atomicAdd(sums + 1, (unsigned long long)t_pess);
        if (t_cnt) atomicAdd(sums + 2, (unsigned long long)t_cnt);
    }
}

// n_slots: the positives an extra interval may hold (n_pos, or the closure's on a held-out set)
int validate(const lec_rank_t* r, const int64_t* rank_sums, const double* ap, int64_t n_slots) {
    return eval_validate(r, r && r->pos_ptr && rank_sums && ap, [&] {
        if (r->n_pos < 0 || r->n_pos > 0x7fffffffLL) return LEC_E_SIZE;
        const lec_recon_extra_t* x = r->extra;
        if (x && x->count != 0) {
            if (x->count < 0 || x->count > n_slots) return LEC_E_SIZE;  // an extra interval holds at least one positive
            if (!x->ptr || !x->lo || !x->hi) return LEC_E_NULL;
        }
        return 0;
    });
}

}  // namespace
}  // namespace lec

extern "C" int64_t lec_rank_workspace_bytes(int64_t n, int64_t n_pos) {
    using namespace lec;
    if (n < 0 || n > 0x7fffffffLL || n_pos < 0 || n_pos > 0x7fffffffLL) return LEC_E_SIZE;
    size_t temp = 0;
    const cudaError_t e = sort_temp_bytes(n, n_pos, temp);
    if (e != cudaSuccess) return -(int64_t)e;
    return (int64_t)(rank_layout(nullptr, n, n_pos).fixed + al256(temp));
}

extern "C" int lec_rank_run_heldout(const lec_rank_t* r, const lec_heldout_t* h, int64_t* rank_sums, double* ap,
                                    int32_t* ranks, void* stream) {
    using namespace lec;
    int err = validate(r, rank_sums, ap, h ? h->n_closure : r ? r->n_pos : 0);
    if (err) return err;
    if (h) {
        if ((err = heldout_validate(h, r->extra && r->extra->count != 0))) return err;
        if (r->n_pos > h->n_closure) return LEC_E_SIZE;
    }
    const RankLayout l = rank_layout(r->workspace, r->n, r->n_pos);
    size_t temp = 0;
    cudaError_t e = sort_temp_bytes(r->u_end - r->u_begin, r->n_pos, temp);
    if (e != cudaSuccess) return (int)e;
    if ((int64_t)(l.fixed + temp) > r->workspace_bytes) return LEC_E_SIZE;
    cudaStream_t st = (cudaStream_t)stream;
    struct Events {  // stage timing (stage_ms != NULL only)
        cudaEvent_t ev[5] = {};
        ~Events() { for (auto& v : ev) if (v) cudaEventDestroy(v); }
    } t;
    if (r->stage_ms) {
        for (auto& v : t.ev)
            if ((e = cudaEventCreate(&v)) != cudaSuccess) return (int)e;
    }
    auto mark = [&](int i) {
        if (r->stage_ms) cudaEventRecord(t.ev[i], st);
    };
    e = cudaMemsetAsync(rank_sums, 0, 3 * sizeof(int64_t), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(l.cnt, 0, (size_t)(static_cast<char*>(l.temp) - reinterpret_cast<char*>(l.cnt)), st);
    if (e != cudaSuccess) return (int)e;
    const int64_t rows = r->u_end - r->u_begin;
    int rc = 0;
    if (rows > 0 && r->n_pos > 0) {
        const lec_recon_extra_t* x = (r->extra && r->extra->count != 0) ? r->extra : nullptr;
        mark(0);
        rank_apex_kernel<<<1, kRankPrepThreads, 0, st>>>(r->pos_ptr, r->u_begin, r->u_end, l.apex, l.napex);
        ++g_launches;
        if (x && !h) {
            rank_xcum_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(r->tin, r->tout, x->ptr, x->lo, x->hi, r->u_begin,
                                                                        r->u_end, l.xcum);
            ++g_launches;
        }
        FastArgs a{};
        a.labels = r->rows; a.images = r->rows; a.L = r->n; a.N = r->n; a.D = r->D; a.K = r->K; a.k = 1;
        a.ld = r->ld; a.u_begin = 0; a.u_end = rows;
        a.tin = r->tin; a.tout = r->tout;
        if (x) { a.xptr = x->ptr; a.xlo = x->lo; a.xhi = x->hi; }
        a.rapex = l.apex; a.rnapex = l.napex; a.rpos = r->pos_ptr; a.rxcum = h ? h->xcum : l.xcum;
        a.rkey = l.key_in; a.rval = l.val_in; a.rsorted = l.key_out; a.rcnt = l.cnt; a.req = l.eq;
        if (h) { a.hptr = h->closure_ptr; a.hmap = h->slot_map; }
        rc = h ? eval_launch<Pass::RankKeysHeld>(r->geom, a, st) : eval_launch<Pass::RankKeys>(r->geom, a, st);
        if (rc) return rc;
        mark(1);
        size_t tb = temp;
        e = cub::DeviceSegmentedRadixSort::SortPairs(l.temp, tb, l.key_in, l.key_out, l.val_in, l.val_out, (int)r->n_pos,
                                                     (int)rows, r->pos_ptr + r->u_begin, r->pos_ptr + r->u_begin + 1, 0,
                                                     kRankKeyBits, st);
        if (e != cudaSuccess) return (int)e;
        mark(2);
        rc = eval_launch<Pass::RankCounts>(r->geom, a, st);
        if (rc) return rc;
        mark(3);
        rank_finish_kernel<<<kRankFinishBlocks, kRankFinishThreads, 0, st>>>(
            r->pos_ptr, l.apex, l.napex, l.key_out, l.val_out, l.cnt, l.eq,
            reinterpret_cast<unsigned long long*>(rank_sums), ap, ranks);
        ++g_launches;
        mark(4);
        if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
    }
    if (r->stage_ms) {
        if (rows > 0 && r->n_pos > 0) {
            if ((e = cudaEventSynchronize(t.ev[4])) != cudaSuccess) return (int)e;
            for (int i = 0; i < 4; ++i) cudaEventElapsedTime(r->stage_ms + i, t.ev[i], t.ev[i + 1]);
        } else {
            for (int i = 0; i < 4; ++i) r->stage_ms[i] = 0.f;
        }
    }
    return 0;
}

extern "C" int lec_rank_run(const lec_rank_t* r, int64_t* rank_sums, double* ap, int32_t* ranks, void* stream) {
    return lec_rank_run_heldout(r, nullptr, rank_sums, ap, ranks, stream);
}
